// lev_bvfused.cu -- Kb, the unit-cost n-best fast path as ONE kernel: lengths, run detection,
// token -> match-mask tables and Myers' bit-vector recurrence, lane = pair, straight from the
// raw sequence-first tokens to the (H', N) output rows.
//
// The hash look-up of hypothesis token i feeds the Myers step of row i directly: the look-up's
// shared-memory latency hides behind the ~45 ALU instructions of the previous row's step, and
// no per-token intermediate goes through global memory (DESIGN §9).  Per warp (32 consecutive
// pairs = 4 runs of an 8-best batch):
//
//   A  one coalesced pass over the reference columns: runs of identical references (each lane
//      compares with its left neighbour), first eos, "needs 64-bit compares" (lev_bvf_scan)
//   B  per run, its lanes build ONE bucketed hash table token -> first-claimed position
//      (lev_bv_build_table, lev_bitvec.cuh), then set, for every reference position, its bit in
//      the match mask Peq[position] of the run (shared-memory atomicOr)
//   C  every lane streams ITS hypothesis column (rows of 32 neighbouring pairs: one coalesced
//      256-byte load per row, two halves of 8 rows in flight), and per token: hash -> 128-bit
//      read of the bucket's keys -> position (lev_bv_row) -> 128-bit read of Peq -> Myers step ->
//      one output row (32 neighbouring pairs: one 128-byte store).  The eos / length logic of
//      SM:195-228 and the freezing of SM:286-288 run inside the stream: a lane stops stepping
//      at its first eos, rows beyond become `padding`.
//
// Selection: lev_bv_probe_kernel looks at 16 positions of the references of a sample of 32-pair
// blocks and vetoes (state[3]) when a block holds more than 4 distinct references -- unrelated
// references differ almost everywhere.  After it the decision is final, so the wavefront path's
// stand-by chain forks from there and runs BESIDE this kernel (lev_abi.cu, LevFork).  A block
// the probe did not see (or whose references agree on the probed positions) is still computed
// correctly here: more than 4 runs are taken in several passes, tokens outside int32 by an
// exact-compare loop.
#include "lev_bitvec.cuh"

#ifndef LEV_BVF_WARPS_PER_CTA
#define LEV_BVF_WARPS_PER_CTA 4  // at most: fewer where the tables of that many do not fit (host)
#endif
#ifndef LEV_BVF_CTAS_PER_SM
#define LEV_BVF_CTAS_PER_SM 3  // resident CTAs per SM the launch bounds and the grid are sized for
#endif
// tuning switches (scripts/gpu_ab.sh builds one library per setting)
#ifndef LEV_BVF_NBUF
#define LEV_BVF_NBUF 4  // chunk buffers of the hypothesis stream: loads run NBUF - 1 trips ahead
#endif
#ifndef LEV_BVF_CH
#define LEV_BVF_CH 4  // hypothesis positions per loop trip
#endif
#ifndef LEV_BVF_PF_AHEAD
#define LEV_BVF_PF_AHEAD 32  // rows the L2 prefetch runs ahead of the hypothesis stream
#endif
#ifndef LEV_BVF_PROBE_BLOCKS
#define LEV_BVF_PROBE_BLOCKS 1024  // blocks of 32 pairs the probe samples at most
#endif

// ---- the match-mask table of one pass: M[(R + 1)][NT][W], row R stays zero (no match) ----
template <int W>
__device__ __forceinline__ void lev_bvf_load_eq(const unsigned* row, unsigned (&eq)[W]) {
    if (W == 4) {
        const uint4 e = *reinterpret_cast<const uint4*>(row);
        eq[0] = e.x;
        eq[W > 1 ? 1 : 0] = e.y;
        eq[W > 2 ? 2 : 0] = e.z;
        eq[W > 3 ? 3 : 0] = e.w;
    } else if (W == 2) {
        const uint2 e = *reinterpret_cast<const uint2*>(row);
        eq[0] = e.x;
        eq[W > 1 ? 1 : 0] = e.y;
    } else {
#pragma unroll
        for (int w = 0; w < W; ++w) eq[w] = row[w];
    }
}

// Myers step that also hands back the top words of the horizontal +1 / -1 vectors: their sign
// bits are the change of the score at reference column r.
template <int W>
__device__ __forceinline__ void lev_bvf_step(const unsigned (&eq)[W], unsigned (&pv)[W],
                                             unsigned (&mv)[W], unsigned& up_w, unsigned& down_w) {
    unsigned t[W], sum[W], ph[W], mh[W];
#pragma unroll
    for (int w = 0; w < W; ++w) t[w] = eq[w] & pv[w];
    lev_bv_add<W>(t, pv, sum);
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const unsigned xh = (sum[w] ^ pv[w]) | eq[w];
        ph[w] = mv[w] | ~(xh | pv[w]);
        mh[w] = pv[w] & xh;
    }
    up_w = ph[W - 1];
    down_w = mh[W - 1];
#pragma unroll
    for (int w = W - 1; w >= 0; --w) {
        const unsigned phs = w ? __funnelshift_l(ph[w - 1], ph[w], 1) : ((ph[0] << 1) | 1u);
        const unsigned mhs = w ? __funnelshift_l(mh[w - 1], mh[w], 1) : (mh[0] << 1);
        const unsigned xv = eq[w] | mv[w];
        pv[w] = mhs | ~(xv | phs);
        mv[w] = phs & xv;
    }
}

// A: one coalesced pass over a lane's reference column, 8 positions per half, the two halves'
// loads ping-pong.  Runs of identical references (SM:1426/1439 repeat every reference over its
// n-best list): a lane compares with its left neighbour through ONE shuffle per token -- the low
// words; the high words only matter if some token of the warp is not an int32 value, which is
// found on the way (wide) and settled by a second, rare, pass.  First eos: SM:137-143, 198-218.
struct LevBvfScan {
    int first_eos;  // position of the first eos in my reference column (R: none)
    bool wide;      // my column holds a token outside int32
    bool diff;      // my column differs from my left neighbour's (a run starts at this lane)
};
template <typename TT>
__device__ __forceinline__ LevBvfScan lev_bvf_scan(const LevBvArgs& a, const TT* __restrict__ rsrc,
                                                   const int rst, const int64_t rcol, const int lane) {
    LevBvfScan s;
    s.first_eos = a.R;
    const int prev_col = __shfl_up_sync(LEV_FULL_MASK, (int)rcol, 1);
    const bool other = prev_col != (int)rcol;
    const int eos_lo = (int)a.eos, eos_hi = (int)(a.eos >> 32);
    int dacc = 0, wacc = 0;  // differences to the left neighbour / to a sign extension
    constexpr int DH = 8;
    const int Rm1 = a.R - 1;
    auto observe = [&](const TT (&buf)[DH], int t0) {
        unsigned eos_bits = 0;
#pragma unroll
        for (int k = 0; k < DH; ++k) {
            const int64_t x = (int64_t)buf[k];
            const int lo = (int)x, hi = (int)(x >> 32);
            dacc |= lo ^ __shfl_up_sync(LEV_FULL_MASK, lo, 1);
            int e = lo ^ eos_lo;
            if (sizeof(TT) == 8) {
                wacc |= hi ^ (lo >> 31);
                e |= hi ^ eos_hi;
            }
            eos_bits |= e == 0 ? (1u << k) : 0u;
        }
        // positions past R repeat position R - 1 (clamped loads): mask them out
        const int live = a.R - t0;
        if (live < DH) eos_bits &= live > 0 ? (1u << live) - 1u : 0u;
        if (eos_bits != 0 && s.first_eos == a.R) s.first_eos = t0 + __ffs((int)eos_bits) - 1;
    };
    // the column is read in order, DH rows at a time: a running pointer and `row k of the batch`
    // offsets; only the batches that reach past the last row clamp per load
    const TT* __restrict__ rp = rsrc;
    int tl = 0;  // first row of the next batch
    auto ld_batch = [&](TT (&buf)[DH]) {
        if (tl + DH <= a.R) {  // (warp-uniform)
#pragma unroll
            for (int k = 0; k < DH; ++k) buf[k] = rp[(int64_t)k * rst];
            rp += (int64_t)DH * rst;
        } else {
#pragma unroll
            for (int k = 0; k < DH; ++k) {
                const int t = tl + k;
                buf[k] = rsrc[(int64_t)(t < Rm1 ? t : Rm1) * rst];
            }
        }
        tl += DH;
    };
    TT bufA[DH], bufB[DH];
    ld_batch(bufA);
#pragma unroll 1
    for (int t0 = 0; t0 < a.R; t0 += 2 * DH) {
        ld_batch(bufB);
        observe(bufA, t0);
        ld_batch(bufA);
        observe(bufB, t0 + DH);
    }
    if (!a.has_eos) s.first_eos = a.R;
    s.wide = wacc != 0;
    if (sizeof(TT) == 8 && __any_sync(LEV_FULL_MASK, s.wide)) {
        // rare: equal low words prove nothing next to a token outside int32 -- compare the high
        // words too (cached re-read)
#pragma unroll 1
        for (int t = 0; t < a.R; ++t) {
            const int hi = (int)((int64_t)rsrc[(int64_t)t * rst] >> 32);
            dacc |= hi ^ __shfl_up_sync(LEV_FULL_MASK, hi, 1);
        }
    }
    s.diff = dacc != 0 && other;
    return s;
}

// KIND: 0 = final value, 1 = prefix rows, 2 = prefix rows with exclude_last.
// One block of 32 consecutive pairs, one warp.  Lanes past the batch shadow its last pair: they
// compute -- and store -- exactly what that pair's own lane does, so nothing in here is
// predicated on "is my pair real".
template <typename TT, int W, int KIND>
__device__ __forceinline__ void lev_bvf_block(const LevBvArgs& a, uint4* keys4, unsigned* M,
                                              const int nb, const int tab_words,
                                              const int64_t block, const int64_t next_block,
                                              const bool first_block, const int lane) {
    constexpr int NT = LEV_BV_NT;
    constexpr bool PREFIX = KIND != 0, EXCL = KIND == 2;
    // hypothesis positions per loop trip: small on purpose -- the stream loop (~100 instructions
    // per position) has to stay inside the instruction caches next to the scan and build loops
    // of the warps that are in another phase (ncu: no_instruction was the top stall at 8)
    constexpr int CH = LEV_BVF_CH;
    const int64_t pair = block * 32 + lane;
    const int64_t pc = pair < a.P ? pair : (int64_t)a.P - 1;
    const int64_t rcol = pc / a.ref_group;
    const TT* __restrict__ rsrc = reinterpret_cast<const TT*>(a.ref) + rcol;
    const TT* __restrict__ hsrc = reinterpret_cast<const TT*>(a.hyp) + pc;
    const int rst = (int)a.ref_st, hst = (int)a.hyp_st;
    const int Z = a.R;
    const int eos_lo = (int)a.eos, eos_hi = (int)(a.eos >> 32);
    const int H = a.H, Hm1 = a.H - 1;
    // The rows of 32 neighbouring pairs are 1 or 2 cache lines: ONE prefetch instruction of the
    // warp covers 16 rows of a block (lane -> row, line).  Used 32 rows ahead of the hypothesis
    // stream, and -- from the middle of a block's stream -- for the first rows of the NEXT block
    // this warp will take, so that its reference scan starts on L2 hits instead of DRAM latency.
    constexpr int LINE = 128 / (int)sizeof(TT);
    auto prefetch16 = [&](const void* base, int64_t first_col, int64_t ncols, int64_t stride, int t_first,
                          int nrows) {
        const int64_t col = first_col + (lane >> 4) * LINE;
        const int t = t_first + (lane & 15);
        if (nrows > 0)
            lev_prefetch_l2(reinterpret_cast<const TT*>(base) + (col < ncols ? col : ncols - 1) +
                            (int64_t)(t < nrows - 1 ? t : nrows - 1) * stride);
    };
    auto prefetch_hyp = [&](int64_t blk, int t_first) { prefetch16(a.hyp, blk * 32, a.P, hst, t_first, H); };
    // (the two divisions are taken once per block, not once per prefetch inside the stream loop)
    const int64_t ref_ncols = (a.P + a.ref_group - 1) / a.ref_group;
    const int64_t next_ref_col = next_block >= 0 ? (next_block * 32) / a.ref_group : 0;
    auto prefetch_ref = [&](int64_t first_col, int t_first) {
        prefetch16(a.ref, first_col, ref_ncols, rst, t_first, a.R);
    };
    if (first_block) {  // (later blocks were announced by the block before them)
        for (int t = 0; t < a.R; t += 16) prefetch_ref((block * 32) / a.ref_group, t);
        prefetch_hyp(block, 0);
        prefetch_hyp(block, 16);
    }

    // ---- A: my reference column -----------------------------------------------------------
    const LevBvfScan scan = lev_bvf_scan<TT>(a, rsrc, rst, rcol, lane);
    const LevBvRuns runs = lev_bv_runs(!scan.diff, lane);
    int rlen = a.R;
    int myflags = 0;
    if (scan.first_eos < a.R) rlen = scan.first_eos + (a.include_eos ? 1 : 0);
    if (a.has_eos && a.include_eos && scan.first_eos == a.R) myflags |= B200LEV_FLAG_REF_NO_EOS;
    const int o = 32 * W - rlen;  // the reference occupies bits [o, 32 W)
    // SM:352-388 as one branch-free formula per row: v = s * mult, then the correctly rounded
    // v / r (Markstein: q0 = v * y, q0 + y * (v - r * q0)) -- with y = r = 1 that is v itself, so
    // `norm` only chooses the constants; an empty reference under `norm` is 0 for row 0 and 1
    // for every later row (mult 0, bias 1).
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
    const int haseos_m = a.has_eos ? -1 : 0, incl_m = a.include_eos ? -1 : 0;
    int hlen = 0;

#pragma unroll 1
    for (int base = 0; base < runs.count; base += NT) {
        const bool active = runs.index >= base && runs.index < base + NT;
        const int tb = active ? runs.index - base : 0;
        const bool leader = active && runs.lead == lane;
        const int run_pos = lane - runs.lead;

        // ---- B: the run's hash table, then its match masks -----------------------------------
        int seed = 0;
        const int exact = lev_bv_build_table<TT>(a, keys4, nb, rsrc, rst, runs, active, tb, run_pos,
                                                 scan.wide ? 1 : 0, lane, &seed);
        {
            uint4* mz = reinterpret_cast<uint4*>(M);
            for (int i = lane; i < tab_words / 4; i += 32) mz[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        __syncwarp();
        const unsigned hmul = lev_bv_mult(seed);
        const unsigned nmul = hmul * (0u - (1u << a.slots_log2));  // v * nmul = -(x << s)
        const int hshift = 32 - a.slots_log2;
        // my run's slice of the tables: bucket b is keys_tb[b * NT]
        const uint4* __restrict__ keys_tb = keys4 + tb;
        const unsigned* __restrict__ M_tb = M + tb * W;
        if (active && !exact) {
            for (int t0 = run_pos; t0 < rlen; t0 += 8 * runs.len) {
                int vv[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    vv[k] = (t0 + k * runs.len < rlen) ? (int)rsrc[(int64_t)(t0 + k * runs.len) * rst] : 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int t = t0 + k * runs.len;
                    if (t >= rlen) break;
                    const unsigned v = (unsigned)vv[k];
                    // the rule the hypothesis look-ups use too
                    const unsigned u = lev_bv_row(keys_tb[(int)((v * hmul) >> hshift) * NT], v * nmul, Z);
                    const int b = t + o;
                    atomicOr(&M[(u * NT + tb) * W + (b >> 5)], 1u << (b & 31));
                }
            }
        }
        if (leader && exact) {
            // rare: reference tokens outside int32, or no overflow-free table: the row of a
            // position is its first occurrence, found by exact comparison
            for (int j = 0; j < rlen; ++j) {
                const TT x = rsrc[(int64_t)j * rst];
                int u = j;
                for (int e = 0; e < j; ++e)
                    if (rsrc[(int64_t)e * rst] == x) {
                        u = e;
                        break;
                    }
                const int b = j + o;
                M[(u * NT + tb) * W + (b >> 5)] |= 1u << (b & 31);
            }
        }
        __syncwarp();

        // ---- C: my hypothesis column, one position per output row ------------------------------
        // Position t emits output row t (a value if the hypothesis reaches that far, else
        // `padding`), then steps to row t + 1 with token t.  Everything per-lane is a mask (0 / -1)
        // or a select: no divergent branch in the stream.  A lane whose hypothesis has ended
        // keeps stepping on garbage; nothing of it is used (its rows are padding, its final
        // score and length are masked).
        unsigned pv[W], mv[W];
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int lo = 32 * w;
            pv[w] = o <= lo ? ~0u : (o >= lo + 32 ? 0u : (~0u << (o - lo)));
            mv[w] = 0u;
        }
        int score = rlen;            // FINAL: the running distance
        float scoref = (float)rlen;  // PREFIX: the same in fp32 (exact: < 2^24), FMA pipe
        int live_m = active ? -1 : 0;  // my hypothesis has not ended yet
        int prev_m = -1;               // token t - 1 was inside it (row 0: always)
        int nin = 0;                   // tokens inside = the hypothesis length (SM:195-228)
        float prev_val = PREFIX ? value_of(scoref, 0.0f) : 0.0f;
        float* __restrict__ orow = a.out + pc;

        // (a trip may run past the last token, t >= H: such a position only emits its row)
        auto position = [&](const TT tok, const int t, auto&& row_of) {
            const int64_t x = (int64_t)tok;
            const int v = (int)x, hi = (int)(x >> 32);
            int e = v ^ eos_lo;
            if (sizeof(TT) == 8) e |= hi ^ eos_hi;
            const int eos_m = e == 0 ? haseos_m : 0;
            const int has_tok = t < H ? -1 : 0;  // (warp-uniform)
            // the hypothesis ends before its first eos, or with it (include_eos)
            const int in_m = live_m & (incl_m | ~eos_m) & has_tok;
            live_m &= ~eos_m & has_tok;
            nin -= in_m;
            if (PREFIX) {
                // row t is a value iff t <= h (t < h with exclude_last: token t must exist)
                const int c_m = EXCL ? in_m : prev_m;
                lev_st_f32_if(t < a.Hout, orow, c_m != 0 ? prev_val : a.padding);
                orow += a.out_si;
                prev_m = in_m;
            }
            unsigned eq[W];
            lev_bvf_load_eq<W>(row_of(x, v, hi), eq);
            unsigned up_w, down_w;
            lev_bvf_step<W>(eq, pv, mv, up_w, down_w);
            const int up_s = (int)up_w >> 31, down_s = (int)down_w >> 31;  // -1: the score moves
            if (PREFIX) {
                // +1.0f / -1.0f / 0 assembled from the two sign masks
                const unsigned bits = ((unsigned)(up_s | down_s) & 0x3f800000u) | ((unsigned)down_s & 0x80000000u);
                scoref += __int_as_float((int)bits);
                prev_val = value_of(scoref, bias);
            } else {
                score += (down_s - up_s) & in_m;
            }
        };
        // the run's table: one 128-bit read of the bucket's keys settles a look-up -- no probe
        // loop; a token no way holds reads row Z (= the all-zero row)
        auto row_hashed = [&](int64_t, int v, int hi) -> const unsigned* {
            const unsigned uv = (unsigned)v;
            unsigned u = lev_bv_row(keys_tb[(int)((uv * hmul) >> hshift) * NT], uv * nmul, Z);
            if (sizeof(TT) == 8) u = hi != (v >> 31) ? (unsigned)Z : u;  // not an int32 token: no key holds it
            return M_tb + u * (NT * W);
        };
        auto row_exact = [&](int64_t x, int, int) -> const unsigned* {
            int u = Z;
            for (int e = 0; e < rlen; ++e)
                if ((int64_t)rsrc[(int64_t)e * rst] == x) {
                    u = e;
                    break;
                }
            return M_tb + u * (NT * W);
        };

        // the stream: every lane of the warp iterates (the vote below is warp-wide), the lanes
        // of this pass that have a table work
        const bool fast = active && !exact;
        const int T_end = PREFIX ? (a.Hout > H ? a.Hout : H) : H;  // positions to visit
        int tdone = 0;  // positions (= output rows) done by the stream
        if (H > 0 && __any_sync(LEV_FULL_MASK, fast)) {
            // the column is read strictly in order, CH rows at a time: a running pointer and
            // `row k of the chunk` offsets (one IMAD.WIDE per load instead of a clamp and a 64-bit
            // multiply-add); only the chunks that reach past the last row clamp per load
            const TT* __restrict__ hp = hsrc;
            int tl = 0;  // first row of the next chunk
            auto ld_chunk = [&](TT (&buf)[CH]) {
                if (tl + CH <= H) {  // (warp-uniform)
#pragma unroll
                    for (int k = 0; k < CH; ++k)
                        buf[k] = lev_ldg_stream(hp + (int64_t)k * hst);
                    hp += (int64_t)CH * hst;
                } else {
#pragma unroll
                    for (int k = 0; k < CH; ++k) {
                        const int t = tl + k;
                        buf[k] = lev_ldg_stream(hsrc + (int64_t)(t < Hm1 ? t : Hm1) * hst);
                    }
                }
                tl += CH;
            };
            // NBUF chunk buffers rotate: the loads of a chunk are issued NBUF - 1 trips before its
            // tokens are looked up (4 buffers: 12 positions, > 1000 issue slots of this warp); the
            // rotation's register moves run on the FMA pipe
            constexpr int NBUF = LEV_BVF_NBUF;
            TT buf[NBUF][CH];
#pragma unroll
            for (int b = 0; b < NBUF - 1; ++b) ld_chunk(buf[b]);
            int t0 = 0;
#pragma unroll 1
            for (; t0 < T_end; t0 += CH) {
                if ((t0 & 15) == 0) {
                    prefetch_hyp(block, t0 + LEV_BVF_PF_AHEAD);
                    if (next_block >= 0) {  // announce the next block of this warp
                        if (t0 < a.R) prefetch_ref(next_ref_col, t0);
                        if (t0 < 32) prefetch_hyp(next_block, t0);
                    }
                }
                ld_chunk(buf[NBUF - 1]);
                if (fast) {
#pragma unroll
                    for (int k = 0; k < CH; ++k) position(buf[0][k], t0 + k, row_hashed);
                }
#pragma unroll
                for (int b = 0; b < NBUF - 1; ++b)
#pragma unroll
                    for (int k = 0; k < CH; ++k) buf[b][k] = buf[b + 1][k];
                // every hypothesis of this pass has ended: the remaining rows are padding
                if ((t0 & 12) == 12 && !__any_sync(LEV_FULL_MASK, fast && live_m != 0)) {
                    t0 += CH;
                    break;
                }
            }
            if (fast) tdone = t0 < T_end ? t0 : T_end;
        }
        if (active && exact) {
#pragma unroll 1
            for (int t = 0; t < T_end; ++t)
                position(hsrc[(int64_t)(t < Hm1 ? t : (Hm1 > 0 ? Hm1 : 0)) * hst], t, row_exact);
            tdone = T_end;
        }
        if (active) {
            if (PREFIX) {
                // rows the stream did not reach (it ended early, or there are no tokens at all):
                // row `tdone` still counts when the token before it did; the rest is padding
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
            hlen = nin;
            if (a.has_eos && a.include_eos && live_m != 0) myflags |= B200LEV_FLAG_HYP_NO_EOS;
            if (!PREFIX) {  // SM:390-405
                float val = __fmul_rn((float)score, a.mult);
                if (a.norm) val = (rlen == 0) ? (hlen > 0 ? 1.0f : 0.0f) : val / (float)rlen;
                a.out[pc] = val;
            }
        }
    }
    if (next_block >= 0) {  // whatever of the next block's first rows the stream did not announce
        for (int t = 0; t < a.R; t += 16) prefetch_ref(next_ref_col, t);
        prefetch_hyp(next_block, 0);
        prefetch_hyp(next_block, 16);
    }
    a.hyp_len[pc] = hlen;
    if (pc % a.ref_group == 0) a.ref_len[rcol] = rlen;
    if (a.norm && rlen == 0) myflags |= B200LEV_FLAG_EMPTY_REF;  // SM:360-366, 397-404
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) myflags |= __shfl_xor_sync(LEV_FULL_MASK, myflags, d);
    if (lane == 0 && myflags != 0 && a.flags != nullptr) atomicOr(a.flags, myflags);
    __syncwarp();  // the next block of this warp reuses the tables
}

// Warps are independent: each takes the block of 32 pairs of its own index, then claims further
// blocks from a global counter.  Per warp: keys [nb][NT] uint4 (4 ways), M [(R + 1)][NT][W] words.
template <typename TT, int W, int KIND>
__global__ void __launch_bounds__(32 * LEV_BVF_WARPS_PER_CTA, LEV_BVF_CTAS_PER_SM) lev_bv_fused_kernel(const LevBvArgs a) {
    if (a.check_state && !lev_bv_took(a.state)) return;  // the probe handed the batch back
    LEV_DYN_SMEM(unsigned, smem);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int nb = 1 << a.slots_log2;
    const int tab_words = ((a.R + 1) * W * LEV_BV_NT + 3) & ~3;
    uint4* keys4 = reinterpret_cast<uint4*>(smem + (size_t)warp * (nb * LEV_BV_NT * 4 + tab_words));
    unsigned* M = reinterpret_cast<unsigned*>(keys4 + nb * LEV_BV_NT);
    const int64_t nblocks = ((int64_t)a.P + 31) / 32;
    const int64_t stride = (int64_t)gridDim.x * warps;
    const int64_t first = (int64_t)blockIdx.x * warps + warp;
    // The first block of a warp is its own; further ones are claimed from a counter (zeroed by
    // the probe or a memset), one block AHEAD so that the stream of the current block can
    // announce the next one to L2.  A warp's blocks take different times (ragged hypotheses,
    // table retries): equal shares leave the last warps of an SM running alone at a third of
    // the occupancy.
    int* counter = a.counter;
    auto claim = [&]() -> int64_t {
        int c = 0;
        if (lane == 0) c = atomicAdd(counter, 1);
        c = __shfl_sync(LEV_FULL_MASK, c, 0);
        const int64_t b = stride + c;
        return b < nblocks ? b : -1;
    };
    int64_t block = first < nblocks ? first : -1;
    bool first_block = true;
    while (block >= 0) {
        const int64_t next = claim();
        lev_bvf_block<TT, W, KIND>(a, keys4, M, nb, tab_words, block, next, first_block, lane);
        block = next;
        first_block = false;
    }
}

// ---- the probe: is this an n-best shaped batch? ---------------------------------------------
// One warp per sampled block of 32 pairs: 16 positions, spread over the row, of the 32
// reference columns; more than NT distinct samples -> veto.
template <typename TT>
__global__ void __launch_bounds__(128) lev_bv_probe_kernel(const LevBvArgs a, const int64_t stride,
                                                           const int64_t nsample) {
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x == 0) *a.counter = 0;
    if (s >= nsample) return;
    const int64_t block = s * stride;
    const int64_t pair = block * 32 + lane;
    const int64_t pc = pair < a.P ? pair : (int64_t)a.P - 1;
    const int64_t rcol = pc / a.ref_group;
    const TT* __restrict__ rsrc = reinterpret_cast<const TT*>(a.ref) + rcol;
    const int prev_col = __shfl_up_sync(LEV_FULL_MASK, (int)rcol, 1);
    TT buf[16];
#pragma unroll
    for (int k = 0; k < 16; ++k)  // 16 positions spread over the row (all of it when R <= 16)
        buf[k] = k < a.R ? rsrc[(int64_t)(a.R <= 16 ? k : (int)(((int64_t)k * a.R) >> 4)) * a.ref_st] : (TT)0;
    int dacc = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const int64_t x = (int64_t)buf[k];
        const int lo = (int)x, hi = (int)(x >> 32);
        dacc |= lo ^ __shfl_up_sync(LEV_FULL_MASK, lo, 1);
        if (sizeof(TT) == 8) dacc |= hi ^ __shfl_up_sync(LEV_FULL_MASK, hi, 1);
    }
    const bool starts = lane == 0 || (dacc != 0 && prev_col != (int)rcol);
    if (__popc(__ballot_sync(LEV_FULL_MASK, starts)) > LEV_BV_NT && lane == 0) atomicExch(a.state + 3, 1);
}

// ---- host side ---------------------------------------------------------------------------------
// every resident slot gets a CTA (the warps walk the blocks with a grid stride; a warp of a
// big batch takes 2-3 blocks, and a full machine during the early rounds beats equal shares)
static unsigned lev_bvf_grid(int64_t P, int warps, int per_sm) {
    const int64_t n = (P + 32 * warps - 1) / (32 * warps);
    int64_t cap = (int64_t)148 * per_sm;
    if (const char* e = getenv("B200LEV_BVF_CTAS")) cap = atoll(e) > 0 ? atoll(e) : cap;  // tests
    return (unsigned)(n < cap ? n : cap);
}

template <typename TT, int W>
static void lev_bvf_launch_w(const LevBvArgs& a, cudaStream_t st) {
    const int nb = 1 << a.slots_log2;
    const int tab_words = ((a.R + 1) * W * LEV_BV_NT + 3) & ~3;
    const size_t warp_bytes = sizeof(unsigned) * (size_t)(nb * LEV_BV_NT * 4 + tab_words);
    // as many warps per CTA (up to the launch bounds') as let LEV_BVF_CTAS_PER_SM CTAs share the
    // 228 KB of an SM (1 KB of it reserved per CTA): at R = 128 the 256-bucket tables take 3
    const size_t per_cta = 228 * 1024 / LEV_BVF_CTAS_PER_SM - 1024;
    int warps = (int)(per_cta / warp_bytes);
    warps = warps < 1 ? 1 : (warps > LEV_BVF_WARPS_PER_CTA ? LEV_BVF_WARPS_PER_CTA : warps);
    const size_t smem = warp_bytes * warps;
    const dim3 grid(lev_bvf_grid(a.P, warps, LEV_BVF_CTAS_PER_SM)), block(32 * warps);
    auto go = [&](auto kern) {
        if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        lev_launch(kern, grid, block, smem, st, a);
    };
    if (a.mode != LEV_MODE_PREFIX)
        go(lev_bv_fused_kernel<TT, W, 0>);
    else if (!a.exclude_last)
        go(lev_bv_fused_kernel<TT, W, 1>);
    else
        go(lev_bv_fused_kernel<TT, W, 2>);
}

template <typename TT>
static void lev_bvf_launch_t(const LevBvArgs& a, cudaStream_t st) {
    switch ((a.R + 31) / 32) {
        case 1: lev_bvf_launch_w<TT, 1>(a, st); break;
        case 2: lev_bvf_launch_w<TT, 2>(a, st); break;
        case 3: lev_bvf_launch_w<TT, 3>(a, st); break;
        default: lev_bvf_launch_w<TT, 4>(a, st); break;
    }
}

bool lev_bvfused_supports(int elem_bytes) {
    return elem_bytes == 8 || elem_bytes == 4 || elem_bytes == 2 || elem_bytes == 1;
}

// `a` as lev_bitvec_launch fills it.  With a.check_state the probe runs first and `after_probe`
// (a cudaEvent_t, may be NULL) is recorded behind it: the veto is final from there on.
int lev_bvfused_launch(const LevBvArgs& a, int elem_bytes, cudaStream_t st, void* after_probe) {
    if (a.check_state) {
        const int64_t nblocks = ((int64_t)a.P + 31) / 32;
        const int64_t stride = (nblocks + LEV_BVF_PROBE_BLOCKS - 1) / LEV_BVF_PROBE_BLOCKS;
        const int64_t nsample = (nblocks + stride - 1) / stride;
        const dim3 grid((unsigned)((nsample + 3) / 4)), block(128);
        lev_prof_begin(LEV_PROF_BV_PROBE, st);
        switch (elem_bytes) {
            case 8: lev_launch(lev_bv_probe_kernel<int64_t>, grid, block, 0, st, a, stride, nsample); break;
            case 4: lev_launch(lev_bv_probe_kernel<int32_t>, grid, block, 0, st, a, stride, nsample); break;
            case 2: lev_launch(lev_bv_probe_kernel<int16_t>, grid, block, 0, st, a, stride, nsample); break;
            default: lev_launch(lev_bv_probe_kernel<int8_t>, grid, block, 0, st, a, stride, nsample); break;
        }
        lev_prof_end(LEV_PROF_BV_PROBE, st);
        const int rc = lev_check_cuda("lev_bv_probe_kernel");
        if (rc) return rc;
    }
    if (!a.check_state && cudaMemsetAsync(a.counter, 0, sizeof(int), st) != cudaSuccess) return lev_check_cuda("memset");
#ifndef B200LEV_EMU
    if (after_probe != nullptr && cudaEventRecord((cudaEvent_t)after_probe, st) != cudaSuccess)
        return lev_check_cuda("cudaEventRecord");
#else
    (void)after_probe;
#endif
    lev_prof_begin(LEV_PROF_BV_DP, st);
    switch (elem_bytes) {
        case 8: lev_bvf_launch_t<int64_t>(a, st); break;
        case 4: lev_bvf_launch_t<int32_t>(a, st); break;
        case 2: lev_bvf_launch_t<int16_t>(a, st); break;
        default: lev_bvf_launch_t<int8_t>(a, st); break;
    }
    lev_prof_end(LEV_PROF_BV_DP, st);
    return lev_check_cuda("lev_bv_fused_kernel");
}
