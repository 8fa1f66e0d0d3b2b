// lev_bvshort.cu -- unit costs, SHORT references (R <= 64), any batch: one LANE per pair, the
// reference in registers, straight from the raw sequence-first tokens to the output.
//
// Short pairs are where the wavefront path pays most for its preparation: on the bulk-scoring
// shape (BASELINE config 4: a million pairs of <= 30 tokens) packing the two token tensors into
// pair-major tables, bucketing the pairs by length and the stand-by launches take as long as
// the DP itself (0.22 of 0.42 ms), and on config 1 (T ~ 50) two thirds of the call.  A
// sequence-first (T, N) tensor is already "position-major, pair-minor": lane l of a warp
// reading tok[t][n0 + l] is one coalesced row, so with lane = pair nothing has to be
// transposed, sorted or staged, and there is no shared memory at all (high occupancy):
//
//   * the lane loads its reference column into registers (<= 64 tokens, their low words; a
//     token outside int32 anywhere in the warp's pairs sends the warp to an exact 64-bit
//     compare loop instead);
//   * per hypothesis token the match mask Eq of Myers' recurrence is built by comparing the
//     token with every reference register, two positions per instruction (16-bit halves,
//     lev_bvs_neq16): no table, no hashing, unrelated references cost the same as shared ones;
//   * one Myers step (1 or 2 words, reference LEFT-aligned: bit j = position j) per hypothesis
//     row; prefix modes read the score at bit r - 1 after every step, the final mode freezes the
//     column state at the lane's last counted token and reads the distance off it once
//     (population counts); eos / length logic (SM:195-228), freezing (SM:286-288), scaling,
//     exact division by r and padding exactly as in lev_bvfused.cu;
//   * b200lev_final_sums: the totals of the bulk-scoring command (command_line.py:1135-1147)
//     are accumulated here too, so that call is this one kernel.
//
// Per DP cell that is about one ALU-pipe instruction (the packed wavefront kernel issues 1.5
// and half an FMA-pipe one), and it is the WHOLE call.  Taken unconditionally (no probe, no
// stand-by chain) wherever lev_bitvec_route admits the bit-vector path and R <= 64.
#include "lev_bitvec.cuh"

constexpr int LEV_BVS_WARPS = 4;

template <int P>
struct LevPath {
    static constexpr int value = P;
};

// 16 reference positions per step pair: register k of a word holds the low halves of the tokens
// at positions k (bits 0-15) and k + 16 (bits 16-31).  `nvv` carries the NEGATED low half of the
// hypothesis token in both halves: one DPX instruction (VIADDMNMX.U16x2) adds it to both
// positions modulo 65 536 and clamps each half to 0 / 1 (1 = differs), an integer multiply-add
// (FMA pipe) shifts the pair into the accumulator: after k = 15 .. 0 bit j of the accumulator
// says "position j differs" -- 1 ALU + 1 FMA instruction per TWO positions.
__device__ __forceinline__ unsigned lev_bvs_neg16(unsigned half) { return ((0u - half) & 0xffffu) * 0x00010001u; }
__device__ __forceinline__ unsigned lev_bvs_neq16(const unsigned (&half)[16], unsigned nvv) {
    unsigned acc0 = 0u, acc1 = 0u;  // two chains of 8
#pragma unroll
    for (int k = 15; k >= 8; --k) acc1 = acc1 * 2u + __viaddmin_u16x2(half[k], nvv, 0x00010001u);
#pragma unroll
    for (int k = 7; k >= 0; --k) acc0 = acc0 * 2u + __viaddmin_u16x2(half[k], nvv, 0x00010001u);
    // acc1 holds positions 8..15 / 24..31 at bits 0..7 / 16..23: move them up by 8
    return acc0 + acc1 * 256u;
}

// PH0: the horizontal delta shifted in at column 0 -- 1 where D[i][0] = i, 0 for the infix form
// (D[i][0] = 0)
template <int W, unsigned PH0 = 1u>
__device__ __forceinline__ void lev_bvs_step(const unsigned (&eq)[W], unsigned (&pv)[W],
                                             unsigned (&mv)[W], unsigned (&ph)[W], unsigned (&mh)[W]) {
    unsigned t[W], sum[W];
#pragma unroll
    for (int w = 0; w < W; ++w) t[w] = eq[w] & pv[w];
    lev_bv_add<W>(t, pv, sum);
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const unsigned xh = (sum[w] ^ pv[w]) | eq[w];
        ph[w] = mv[w] | ~(xh | pv[w]);
        mh[w] = pv[w] & xh;
    }
#pragma unroll
    for (int w = W - 1; w >= 0; --w) {
        const unsigned phs = w ? __funnelshift_l(ph[w - 1], ph[w], 1) : ((ph[0] << 1) | PH0);
        const unsigned mhs = w ? __funnelshift_l(mh[w - 1], mh[w], 1) : (mh[0] << 1);
        const unsigned xv = eq[w] | mv[w];
        pv[w] = mhs | ~(xv | phs);
        mv[w] = phs & xv;
    }
}

// KIND: 0 = final value, 1 = prefix rows, 2 = prefix rows with exclude_last, 3 = infix minimum
// (b200lev_infix: column 0 is 0 on every row, the score at bit r - 1 is tracked as in the prefix
// kinds and its minimum over the counted rows, row 0 included, is the value).
// command_line.py:1135-1147: the totals of the bulk-scoring command, folded into the kernel that
// produced the values (fp64 sums; of integers when the values are counts, so exact in any order);
// three atomics per CTA.  Kept out of line: inlined, it costs the DP loop above it 18 registers.
__device__ __forceinline__ void lev_bvs_totals(double sum_out, int sum_len, double* acc, int64_t P, bool first) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        sum_out += __shfl_xor_sync(LEV_FULL_MASK, sum_out, d);
        sum_len += __shfl_xor_sync(LEV_FULL_MASK, sum_len, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(acc + 0, sum_out);
        atomicAdd(acc + 1, (double)sum_len);
        if (first) atomicAdd(acc + 2, (double)P);
    }
}

// CROSS (final mode, b200lev_final_cross): pair p = (g, a, b) of G groups of A x B pairs reads
// reference column p / ref_group (ref_group = B) and hypothesis column g * B + b, both taken once
// per pair; the lanes of a warp then read at most B distinct hypothesis columns per row.
template <typename TT, int W, int KIND, bool CROSS>
__global__ void __launch_bounds__(32 * LEV_BVS_WARPS, W == 1 ? 5 : 4) lev_bv_short_kernel(const LevBvArgs a) {
    constexpr bool PREFIX = KIND == 1 || KIND == 2, EXCL = KIND == 2, INFIX = KIND == 3;
    constexpr int CH = 4;
    const int lane = threadIdx.x & 31;
    const int64_t nblocks = ((int64_t)a.P + 31) / 32;
    const int rst = (int)a.ref_st, hst = (int)a.hyp_st;
    const int R = a.R, H = a.H, Hm1 = a.H - 1;
    const int eos_lo = (int)a.eos, eos_hi = (int)(a.eos >> 32);
    const int haseos_m = a.has_eos ? -1 : 0, incl_m = a.include_eos ? -1 : 0;
    // bulk scoring: this thread's share of the totals lives in shared memory (one slot per
    // thread), not in registers carried through the DP loop
    __shared__ double sums[LEV_BVS_WARPS * 32];
    __shared__ int lens[LEV_BVS_WARPS * 32];
    if (KIND == 0) {
        sums[threadIdx.x] = 0.0;
        lens[threadIdx.x] = 0;
    }
    for (int64_t block = (int64_t)blockIdx.x * LEV_BVS_WARPS + (threadIdx.x >> 5); block < nblocks;
         block += (int64_t)gridDim.x * LEV_BVS_WARPS) {
        // lanes past the batch shadow its last pair (they compute and store the same values)
        const int64_t pair = block * 32 + lane;
        const int64_t pc = pair < a.P ? pair : (int64_t)a.P - 1;
        const int64_t rcol = pc / a.ref_group;
        const int64_t hcol =
            CROSS ? (int64_t)((int)pc / a.cross_ab * a.cross_b + (int)pc % a.cross_b) : pc;
        const TT* __restrict__ rsrc = reinterpret_cast<const TT*>(a.ref) + rcol;
        const TT* __restrict__ hsrc = reinterpret_cast<const TT*>(a.hyp) + hcol;

        // ---- my reference column -> registers (low and high halves of the tokens, packed two
        // positions per register); its length; does it need 64-bit compares; do its tokens sit
        // in one 65 536-wide window (then the low halves alone decide equality) -----------------
        // (the high halves are kept for one-word references only: with two words they would push
        // the kernel into spills, and a warp whose tokens leave the window compares exactly instead)
        constexpr bool HAVE_HI = W == 1;
        unsigned rlo[W][16], rhi[HAVE_HI ? W : 1][16];
        int first_eos = R;
        int wacc = 0;
        unsigned outside = 0u;  // some reference token is outside [base, base + 65536)
        int base = 0;
        {
            unsigned eos_bits[W];
#pragma unroll
            for (int w = 0; w < W; ++w) {
                eos_bits[w] = 0u;
#pragma unroll
                for (int k = 0; k < 16; ++k) rlo[w][k] = 0u;
            }
            // batches of RB positions: the RB loads are issued back to back (one exposed DRAM
            // latency per batch, not per token), then packed.  The column is walked with a running
            // pointer (a 64-bit add per position instead of a 64-bit multiply-add); positions past
            // R repeat position R - 1: they change neither the window nor the FIRST eos, and bits
            // at or above r are never read
            constexpr int RB = W == 1 ? 16 : 8;  // (two-word references are short of registers)
            const TT* __restrict__ rp = rsrc;
#pragma unroll
            for (int j0 = 0; j0 < 32 * W; j0 += RB) {
                if (j0 < R) {  // (warp-uniform)
                    TT raw[RB];
                    if (j0 + RB < R) {
#pragma unroll
                        for (int k = 0; k < RB; ++k) {
                            raw[k] = *rp;
                            rp += rst;
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < RB; ++k) {
                            raw[k] = *rp;
                            if (j0 + k < R - 1) rp += rst;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < RB; ++k) {
                        const int j = j0 + k;
                        const int64_t x = (int64_t)raw[k];
                        const int lo = (int)x, hi = (int)(x >> 32);
                        if (j == 0) base = lo - 32768;
                        outside |= (unsigned)(lo - base) >> 16;
                        if ((j & 16) == 0)
                            rlo[j >> 5][j & 15] = (unsigned)lo & 0xffffu;
                        else  // the upper half of the register position j - 16 opened
                            rlo[j >> 5][j & 15] = __byte_perm(rlo[j >> 5][j & 15], (unsigned)lo, 0x5410);
                        int e = lo ^ eos_lo;
                        if (sizeof(TT) == 8) {
                            wacc |= hi ^ (lo >> 31);
                            e |= hi ^ eos_hi;
                        }
                        eos_bits[j >> 5] |= e == 0 ? (1u << (j & 31)) : 0u;
                    }
                }
            }
            if (a.has_eos) {
#pragma unroll
                for (int w = W - 1; w >= 0; --w)
                    if (eos_bits[w]) first_eos = 32 * w + __ffs((int)eos_bits[w]) - 1;
            }
        }
        int rlen = R, myflags = 0;
        if (first_eos < R) rlen = first_eos + (a.include_eos ? 1 : 0);
        if (a.has_eos && a.include_eos && first_eos == R) myflags |= B200LEV_FLAG_REF_NO_EOS;
        // row value, branch-free (see lev_bvfused.cu): v = s * mult, then the correctly rounded v / r
        const bool empty_norm = a.norm && rlen == 0;
        const float rr = (a.norm && rlen > 0) ? (float)rlen : 1.0f;
        const float yy = (a.norm && rlen > 0) ? __frcp_rn((float)rlen) : 1.0f;
        const float mult_e = empty_norm ? 0.0f : a.mult;
        const float bias = empty_norm ? 1.0f : 0.0f;
        auto value_of = [&](float s, float b) {
            const float v = __fmaf_rn(s, mult_e, b);
            const float q0 = __fmul_rn(v, yy);
            return __fmaf_rn(__fmaf_rn(-rr, q0, v), yy, q0);
        };
        // the score lives at bit r - 1 (an empty reference: every row costs one insertion)
        const int top = rlen > 0 ? rlen - 1 : 0;
        const int top_sh = top & 31;
        const bool top_hi = W > 1 && top >= 32;
        const unsigned empty_up = (!INFIX && rlen == 0) ? 1u : 0u;

        unsigned pv[W], mv[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            pv[w] = ~0u;
            mv[w] = 0u;
        }
        float scoref = (float)rlen;
        float smin = scoref;  // INFIX: the minimum over the counted rows
        int eos_seen = 0;     // INFIX: an eos among the hypothesis tokens (rows past H clear live_m too)
        int live_m = -1, prev_m = -1, nin = 0;
        float prev_val = PREFIX ? value_of(scoref, 0.0f) : 0.0f;
        float* __restrict__ orow = a.out + pc;
        const bool narrow_warp = !__any_sync(LEV_FULL_MASK, outside != 0u);
        const bool wide_warp = (sizeof(TT) == 8 && __any_sync(LEV_FULL_MASK, wacc != 0)) || (!HAVE_HI && !narrow_warp);

        if (HAVE_HI && !narrow_warp && !wide_warp) {
            // (uncommon) some lane's reference leaves its window: the high halves of the tokens
            // join the compare; they are packed here, from the (cached) column, not in the prologue
            // every warp pays for
#pragma unroll
            for (int k = 0; k < 16; ++k) rhi[0][k] = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int lo = (int)(int64_t)rsrc[(int64_t)(j < R - 1 ? j : R - 1) * rst];
                rhi[0][j & 15] |= ((unsigned)lo >> 16) << (j & 16);
            }
        }
        // PATH 0: every token of the warp's references sits in one 65 536-wide window (low halves
        // decide); 1: low and high halves; 2 (rare): exact compares against the cached column.
        // One copy of the hypothesis loop per path keeps the hot one contiguous in the
        // instruction cache.
        auto position = [&](auto path, const TT tok, const int t) {
            constexpr int PATH = decltype(path)::value;
            const int64_t x = (int64_t)tok;
            const int v = (int)x, hi = (int)(x >> 32);
            int e = v ^ eos_lo;
            if (sizeof(TT) == 8) e |= hi ^ eos_hi;
            const int eos_m = e == 0 ? haseos_m : 0;
            const int has_tok = t < H ? -1 : 0;  // (warp-uniform)
            if (INFIX) eos_seen |= eos_m & has_tok;
            const int in_m = live_m & (incl_m | ~eos_m) & has_tok;
            live_m &= ~eos_m & has_tok;
            nin -= in_m;
            if (PREFIX) {
                const int c_m = EXCL ? in_m : prev_m;
                if (t < a.Hout) *orow = c_m != 0 ? prev_val : a.padding;
                orow += a.out_si;
                prev_m = in_m;
            }
            unsigned eq[W];
#pragma unroll
            for (int w = 0; w < W; ++w) eq[w] = 0u;
            if (PATH == 0) {
                // every reference token of the lane lies in [base, base + 65536): a token in
                // the same window is equal iff the low halves are, one outside equals none
                // (that also covers a 64-bit token outside int32, whose low word is garbage).
                // The compare runs regardless and is masked afterwards: no branch per position
                const unsigned nlo = lev_bvs_neg16((unsigned)v & 0xffffu);
                const bool tok_ok = sizeof(TT) == 8 ? (uint64_t)(x - (int64_t)base) < 65536ull
                                                    : (unsigned)(v - base) < 65536u;
                const unsigned ok_m = tok_ok ? ~0u : 0u;
#pragma unroll
                for (int w = 0; w < W; ++w)
                    if (w == 0 || R > 32) eq[w] = ~lev_bvs_neq16(rlo[w], nlo) & ok_m;
            } else if (PATH == 1) {
                const unsigned nlo = lev_bvs_neg16((unsigned)v & 0xffffu);
                const unsigned nhi = lev_bvs_neg16((unsigned)v >> 16);
                const unsigned ok_m = (sizeof(TT) < 8 || hi == (v >> 31)) ? ~0u : 0u;
#pragma unroll
                for (int w = 0; w < W; ++w)
                    if (w == 0 || R > 32)
                        eq[w] = ~(lev_bvs_neq16(rlo[w], nlo) | lev_bvs_neq16(rhi[HAVE_HI ? w : 0], nhi)) & ok_m;
            } else {
#pragma unroll
                for (int w = 0; w < W; ++w)
                    for (int jj = 0; jj < 32 && 32 * w + jj < rlen; ++jj)
                        if ((int64_t)rsrc[(int64_t)(32 * w + jj) * rst] == x) eq[w] |= 1u << jj;
            }
            unsigned ph[W], mh[W];
            if (PREFIX || INFIX) {
                lev_bvs_step<W, INFIX ? 0u : 1u>(eq, pv, mv, ph, mh);
                const unsigned up = (((top_hi ? ph[W - 1] : ph[0]) >> top_sh) & 1u) | empty_up;
                const unsigned down = ((top_hi ? mh[W - 1] : mh[0]) >> top_sh) & 1u & ~empty_up;
                scoref += __int_as_float((int)(up * 0x3f800000u));
                scoref -= __int_as_float((int)(down * 0x3f800000u));
                if (PREFIX) prev_val = value_of(scoref, bias);
                if (INFIX) smin = (in_m != 0 && scoref < smin) ? scoref : smin;
            } else {
                // FINAL: no score is carried.  The column state (the vertical deltas) freezes at the
                // lane's last counted token, and D[r][h] = h + #(+1 deltas) - #(-1 deltas) among the
                // first r positions is read off it after the loop: 2 selects per word and step
                // instead of 6 instructions of score keeping
                unsigned npv[W], nmv[W];
#pragma unroll
                for (int w = 0; w < W; ++w) {
                    npv[w] = pv[w];
                    nmv[w] = mv[w];
                }
                lev_bvs_step<W>(eq, npv, nmv, ph, mh);
#pragma unroll
                for (int w = 0; w < W; ++w) {
                    pv[w] = (npv[w] & (unsigned)in_m) | (pv[w] & ~(unsigned)in_m);
                    mv[w] = (nmv[w] & (unsigned)in_m) | (mv[w] & ~(unsigned)in_m);
                }
            }
        };

        const int T_end = PREFIX ? (a.Hout > H ? a.Hout : H) : H;
        int tdone = 0;
        if (H > 0) {
            // the hypothesis column is walked CH tokens at a time with a running pointer (rows past
            // H - 1 repeat row H - 1: nothing reads them)
            const TT* __restrict__ hp = hsrc;
            int tl = 0;  // the row `hp` points at
            auto ld_chunk = [&](TT (&buf)[CH]) {
                if (tl + CH < H) {  // (warp-uniform)
#pragma unroll
                    for (int k = 0; k < CH; ++k) {
                        buf[k] = lev_ldg_stream(hp);
                        hp += hst;
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < CH; ++k) {
                        buf[k] = lev_ldg_stream(hp);
                        if (tl + k < Hm1) hp += hst;
                    }
                }
                tl += CH;
            };
            int t0 = 0;
            auto hypothesis = [&](auto path) {
                bool done = false;
                if (W == 1) {
                    // two chunk buffers, rotated by NAME (the loop body is two trips): a chunk is
                    // loaded two trips before it is used and nothing touches it in between -- a
                    // rotation by register moves waits for the loads it moves; more trips per body
                    // would push the loop out of the instruction cache
                    TT bA[CH], bB[CH];
                    ld_chunk(bA);
                    ld_chunk(bB);
                    auto trip = [&](TT (&buf)[CH]) {  // CH positions from `buf`, then its next chunk
                        if (!done) {
#pragma unroll
                            for (int k = 0; k < CH; ++k) position(path, buf[k], t0 + k);
                            ld_chunk(buf);
                            t0 += CH;
                            // every hypothesis of the warp has ended, or the last row is out
                            done = t0 >= T_end || !__any_sync(LEV_FULL_MASK, live_m != 0);
                        }
                    };
#pragma unroll 1
                    while (!done) {
                        trip(bA);
                        trip(bB);
                    }
                } else {
                    // two-word references are short of registers and long on code: one trip per
                    // loop body, the buffers rotate through register moves
                    TT cur[CH], n1[CH], n2[CH];
                    ld_chunk(cur);
                    ld_chunk(n1);
#pragma unroll 1
                    while (!done) {
                        ld_chunk(n2);
#pragma unroll
                        for (int k = 0; k < CH; ++k) position(path, cur[k], t0 + k);
#pragma unroll
                        for (int k = 0; k < CH; ++k) {
                            cur[k] = n1[k];
                            n1[k] = n2[k];
                        }
                        t0 += CH;
                        done = t0 >= T_end || !__any_sync(LEV_FULL_MASK, live_m != 0);
                    }
                }
            };
            if (wide_warp)  // (all three conditions are warp-uniform)
                hypothesis(LevPath<2>{});
            else if (narrow_warp)
                hypothesis(LevPath<0>{});
            else if (HAVE_HI)
                hypothesis(LevPath<1>{});
            tdone = t0 < T_end ? t0 : T_end;
        }
        if (PREFIX) {
            int t = tdone;
            if (t < a.Hout) {
                *orow = (!EXCL && prev_m != 0) ? prev_val : a.padding;
                orow += a.out_si;
                ++t;
            }
            for (; t < a.Hout; ++t) {
                *orow = a.padding;
                orow += a.out_si;
            }
        }
        const int hlen = nin;
        if (a.has_eos && a.include_eos && (INFIX ? eos_seen == 0 : live_m != 0)) myflags |= B200LEV_FLAG_HYP_NO_EOS;
        if (INFIX) a.out[pc] = value_of(rlen > 0 ? smin : 0.0f, 0.0f);  // (an empty reference: 0)
        if (KIND == 0) {  // SM:390-405
            int score = hlen;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const int nb = rlen - 32 * w;  // positions of the reference in this word
                const unsigned m = nb >= 32 ? ~0u : (nb > 0 ? (1u << nb) - 1u : 0u);
                score += __popc(pv[w] & m) - __popc(mv[w] & m);
            }
            float val = __fmul_rn((float)score, a.mult);
            if (a.norm) val = (rlen == 0) ? (hlen > 0 ? 1.0f : 0.0f) : val / (float)rlen;
            a.out[pc] = val;
            if (a.acc != nullptr) {
                if (pair < a.P) {  // (lanes shadowing the last pair do not count twice)
                    sums[threadIdx.x] += (double)val;
                    lens[threadIdx.x] += rlen;
                }
                // the warp's last block: its totals go out from inside the loop (code after the
                // loop costs the loop ~20 registers)
                if (block + (int64_t)gridDim.x * LEV_BVS_WARPS >= nblocks)
                    lev_bvs_totals(sums[threadIdx.x], lens[threadIdx.x], a.acc, a.P,
                                   blockIdx.x == 0 && threadIdx.x < 32);
            }
        }
        a.hyp_len[pc] = hlen;
        if (pc % a.ref_group == 0) a.ref_len[rcol] = rlen;
        if (a.norm && rlen == 0) myflags |= B200LEV_FLAG_EMPTY_REF;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) myflags |= __shfl_xor_sync(LEV_FULL_MASK, myflags, d);
        if (lane == 0 && myflags != 0 && a.flags != nullptr) atomicOr(a.flags, myflags);
    }
}

// ---- host side ---------------------------------------------------------------------------------
bool lev_bvshort_supports(int elem_bytes, int64_t R) {
    const char* e = getenv("B200LEV_BV_SHORT");
    if (e != nullptr && atoi(e) == 0) return false;
    return R >= 1 && R <= 64 && (elem_bytes == 8 || elem_bytes == 4 || elem_bytes == 2 || elem_bytes == 1);
}

template <typename TT, int W>
static void lev_bvs_launch_w(const LevBvArgs& a, cudaStream_t st) {
    int64_t n = ((int64_t)a.P + 32 * LEV_BVS_WARPS - 1) / (32 * LEV_BVS_WARPS);
    int64_t cap = (int64_t)148 * (W == 1 ? 20 : 16);  // whole waves of the resident CTAs (5 / 4 per SM)
    if (const char* e = getenv("B200LEV_BVS_CTAS")) cap = atoll(e) > 0 ? atoll(e) : cap;  // (tests: many blocks per warp)
    const dim3 grid((unsigned)(n < cap ? n : cap)), block(32 * LEV_BVS_WARPS);
    if (a.cross_b > 0)  // (final mode only)
        lev_launch(lev_bv_short_kernel<TT, W, 0, true>, grid, block, 0, st, a);
    else if (a.mode == LEV_MODE_INFIX)
        lev_launch(lev_bv_short_kernel<TT, W, 3, false>, grid, block, 0, st, a);
    else if (a.mode != LEV_MODE_PREFIX)
        lev_launch(lev_bv_short_kernel<TT, W, 0, false>, grid, block, 0, st, a);
    else if (!a.exclude_last)
        lev_launch(lev_bv_short_kernel<TT, W, 1, false>, grid, block, 0, st, a);
    else
        lev_launch(lev_bv_short_kernel<TT, W, 2, false>, grid, block, 0, st, a);
}

int lev_bvshort_launch(const LevBvArgs& a, int elem_bytes, cudaStream_t st) {
    lev_prof_begin(LEV_PROF_BV_DP, st);
    const bool two = a.R > 32;
    switch (elem_bytes) {
        case 8: two ? lev_bvs_launch_w<int64_t, 2>(a, st) : lev_bvs_launch_w<int64_t, 1>(a, st); break;
        case 4: two ? lev_bvs_launch_w<int32_t, 2>(a, st) : lev_bvs_launch_w<int32_t, 1>(a, st); break;
        case 2: two ? lev_bvs_launch_w<int16_t, 2>(a, st) : lev_bvs_launch_w<int16_t, 1>(a, st); break;
        default: two ? lev_bvs_launch_w<int8_t, 2>(a, st) : lev_bvs_launch_w<int8_t, 1>(a, st); break;
    }
    lev_prof_end(LEV_PROF_BV_DP, st);
    return lev_check_cuda("lev_bv_short_kernel");
}
