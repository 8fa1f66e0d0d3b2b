// lev_mask16.cu -- K1m: mask mode (optimal completion, SM:271-278, 319-355) for integer costs,
// PACKED: two pairs per warp, one per 16-bit half of every register, on the 2-wide DPX
// instructions of sm_100 (the cell update of lev_group.cu's packed path).
//
// A warp owns a "duo" of neighbouring pairs (2 d, 2 d + 1).  Each lane holds C adjacent DP
// columns of BOTH pairs (right-aligned per pair, single strip: r + 1 <= 32 C) and the warp is
// skewed over hypothesis rows exactly as in lev_dp.cu.  Two passes over the same DP:
//   A  row minima: per cell one VIMNMX.U16x2 on top of the update, chained along the lanes with
//      the shuffle rhythm of the boundary cell; lane 31 leaves min(row i) of both pairs in shared
//      memory.
//   B  equality: per cell one VIADDMNMX.U16x2 (value + negated row minimum, clamped to 0 / 1) and
//      one IMAD shift the "differs" bits of both pairs into one register; after the C cells the
//      lane drops its two C-bit masks into a per-warp shared-memory sheet [row][lane].
// Then, lane = row, the sheet is turned into the row's bitmap over the reference's DISTINCT
// tokens (ranks from lev_uid_kernel; the sets are tiny, so this enumerates a handful of bits)
// and stored -- the same dbits / umax contract as lev_warp_kernel's chained pass, which keeps
// serving whatever this kernel leaves: references with more than 32 distinct tokens, tokens
// outside one 65 536-wide window, float costs, r + 1 > 256, rows too long for the sheet.
//
// Per two cells: pass A 4 ALU + 1 FMA-pipe instructions, pass B 4 + 2 (lev_dp.cu: 10 and 12).
#include <cstdio>
#include <cstdlib>

#include "lev_common.cuh"

#define LEVM_BIG16 16000
constexpr int LEVM_SHEET_WORDS = 17;  // 32 half-words per row + 1 word: lane = row reads conflict-free

__device__ __forceinline__ unsigned levm_neg2(unsigned a, unsigned b) {  // (-a, -b) mod 65536, packed
    return ((0u - a) & 0xffffu) | ((0u - b) << 16);
}

constexpr int LEVM_RING = 64;  // rows of the sheet: 32 in flight (the skew) + 32 being converted

template <int N>
struct LevmCols {
    static constexpr int value = N;
};

// One pass over the duo's DP with C columns per lane.  PASS 0 leaves the NEGATED row minima of
// both pairs in rowmin_s (what pass 1 adds to a cell to test it); PASS 1 fills the sheet and calls
// convert(first_row) whenever 32 rows of it are complete.
template <int C, int PASS, typename Convert>
__device__ __forceinline__ void levm_pass(const LevParams& p, const int lane, const int rA, const int rB,
                                          const int pairA, const int pairB, const int maxsteps,
                                          const unsigned* __restrict__ nht_s, unsigned* __restrict__ rowmin_s,
                                          unsigned* __restrict__ sheet_s, Convert&& convert) {
    const int32_t* __restrict__ rtA = p.ref_tok + (int64_t)(pairA >= 0 ? pairA / p.ref_group : 0) * p.Rp;
    const int32_t* __restrict__ rtB = p.ref_tok + (int64_t)(pairB >= 0 ? pairB / p.ref_group : 0) * p.Rp;
    const unsigned ins2 = (unsigned)p.ins_i * 0x00010001u, del2 = (unsigned)p.del_i * 0x00010001u;
    const unsigned subc = (unsigned)p.sub_i;
    const unsigned BIG2 = (unsigned)LEVM_BIG16 * 0x00010001u;
    const int j0A = rA - 32 * C + lane * C + 1, j0B = rB - 32 * C + lane * C + 1;
    unsigned v[C], rt[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int jA = j0A + c, jB = j0B + c;
        const unsigned vA = (jA >= 0) ? (unsigned)(jA * p.del_i) : (unsigned)LEVM_BIG16;  // SM:258-263
        const unsigned vB = (jB >= 0) ? (unsigned)(jB * p.del_i) : (unsigned)LEVM_BIG16;
        v[c] = vA | (vB << 16);
        const unsigned tA = (jA >= 1 && pairA >= 0) ? ((unsigned)rtA[jA - 1] & 0xffffu) : 0u;
        const unsigned tB = (jB >= 1 && pairB >= 0) ? ((unsigned)rtB[jB - 1] & 0xffffu) : 0u;
        rt[c] = tA | (tB << 16);
    }
    unsigned pl = BIG2, rmrun = BIG2;
    (void)rmrun;
    unsigned short* __restrict__ sheet16 = reinterpret_cast<unsigned short*>(sheet_s);
    const int nsteps = maxsteps + 31;
    int i = 1 - lane;  // the row this lane updates at step s = 1
    // steps in blocks of 32: after the block that ends with step s0 + 31 the rows up to s0 are
    // complete in every lane
    for (int s0 = 0; s0 < nsteps; s0 += 32) {
        const int nk = nsteps - s0 < 32 ? nsteps - s0 : 32;
#pragma unroll 2
        for (int k = 0; k < nk; ++k, ++i) {
            const unsigned sh = __shfl_up_sync(LEV_FULL_MASK, v[C - 1], 1);
            const unsigned in = (lane == 0) ? BIG2 : sh;
            unsigned dg = pl;
            pl = in;
            unsigned in_rm = BIG2;
            if (PASS == 0) {
                const unsigned sh_rm = __shfl_up_sync(LEV_FULL_MASK, rmrun, 1);
                in_rm = (lane == 0) ? BIG2 : sh_rm;
            }
            if ((unsigned)(i - 1) < (unsigned)maxsteps) {
                const unsigned nht = nht_s[i - 1];  // both pairs' row tokens, negated per half
                unsigned lf = in;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const unsigned up = v[c];
                    const unsigned n01 = __viaddmin_u16x2(rt[c], nht, 0x00010001u);  // 1 = tokens differ
                    const unsigned sb = n01 * subc + dg;                              // SM:293
                    const unsigned t = __viaddmin_s16x2(up, ins2, sb);                // SM:292, 316
                    lf = __viaddmin_s16x2(lf, del2, t);                               // SM:317
                    dg = up;
                    v[c] = lf;
                }
                if (PASS == 0) {  // SM:332-333: running minimum of row i over the columns up to mine
                    unsigned rm = in_rm;
#pragma unroll
                    for (int c = 0; c < C; ++c) rm = __vminu2(rm, v[c]);
                    rmrun = rm;
                    if (lane == 31) rowmin_s[i] = levm_neg2(rm & 0xffffu, rm >> 16);
                } else {  // SM:334, 349-354: which of my cells sit on the row minimum
                    const unsigned nmn = rowmin_s[i];
                    unsigned acc = 0u;
#pragma unroll
                    for (int c = 0; c < C; ++c) acc = acc * 2u + __viaddmin_u16x2(v[c], nmn, 0x00010001u);
                    // bit C - 1 - c of a half of ~acc: cell c equals the minimum; A -> byte 0, B -> byte 1
                    const unsigned eq = ~acc & (((1u << C) - 1u) * 0x00010001u);
                    sheet16[(i & (LEVM_RING - 1)) * (2 * LEVM_SHEET_WORDS) + lane] =
                        (unsigned short)__byte_perm(eq, 0u, 0x4420);
                }
            }
        }
        if (PASS == 1 && s0 >= 32 && nk == 32) {
            // rows s0 - 31 .. s0 are complete (lane 31 has just done row s0): 32 rows, lane = row
            __syncwarp();
            convert(s0 - 31);
            __syncwarp();
        }
    }
    if (PASS == 1) {  // the rows the loop did not flush
        __syncwarp();
        const int full = nsteps / 32;                      // whole blocks of steps
        const int flushed = full >= 2 ? 32 * (full - 1) : 0;  // rows 1 .. flushed are out
        for (int first = flushed + 1; first <= maxsteps; first += 32) convert(first);
    }
}

template <int CMAX>
__global__ void __launch_bounds__(256) lev_mask16_kernel(const LevParams p, const int Hs) {
    LEV_DYN_SMEM(unsigned, smem);
    if (!lev_mask16_tokens_ok(p.wide_flag)) return;  // lev_warp_kernel keeps the whole batch
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int per_warp = Hs * 2 + LEVM_RING * LEVM_SHEET_WORDS + (2 * 32 * CMAX) / 4;
    unsigned* nht_s = smem + (size_t)warp * per_warp;  // [Hs]  negated row tokens of both pairs
    unsigned* rowmin_s = nht_s + Hs;                    // [Hs]  negated row minima of both pairs
    unsigned* sheet_s = rowmin_s + Hs;                  // [64][17] equality masks, [row & 63][lane]
    unsigned char* rank_s = reinterpret_cast<unsigned char*>(sheet_s + LEVM_RING * LEVM_SHEET_WORDS);  // [2][32 CMAX]
    const int nduo = (p.P + 1) / 2;
    for (int duo = blockIdx.x * wpc + warp; duo < nduo; duo += gridDim.x * wpc) {
        int pairA = 2 * duo, pairB = 2 * duo + 1;
        if (pairB >= p.P) pairB = -1;
        // a pair whose reference has more than 32 distinct tokens stays with lev_warp_kernel
        if (!lev_mask16_takes(p, pairA)) pairA = -1;
        if (pairB >= 0 && !lev_mask16_takes(p, pairB)) pairB = -1;
        if (pairA < 0 && pairB < 0) continue;
        const int refA = pairA >= 0 ? pairA / p.ref_group : 0, refB = pairB >= 0 ? pairB / p.ref_group : 0;
        const int rA = pairA >= 0 ? p.ref_len[refA] : 0, rB = pairB >= 0 ? p.ref_len[refB] : 0;
        const int hA = pairA >= 0 ? p.hyp_len[pairA] : 0, hB = pairB >= 0 ? p.hyp_len[pairB] : 0;
        const int stepsA = p.exclude_last ? (hA > 0 ? hA - 1 : 0) : hA;  // SM:286-288
        const int stepsB = p.exclude_last ? (hB > 0 ? hB - 1 : 0) : hB;
        const int maxsteps = stepsA > stepsB ? stepsA : stepsB;
        {
            const int32_t* __restrict__ htA = p.hyp_tok + (int64_t)(pairA >= 0 ? pairA : 0) * p.Hp;
            const int32_t* __restrict__ htB = p.hyp_tok + (int64_t)(pairB >= 0 ? pairB : 0) * p.Hp;
            // (both rows run to the longer pair's length: the rows past a pair's own are never read back)
            for (int i = lane; i < maxsteps; i += 32)
                nht_s[i] = levm_neg2((unsigned)htA[i] & 0xffffu, (unsigned)htB[i] & 0xffffu);
            const int32_t* __restrict__ uA = p.uid + (int64_t)refA * p.Rp;
            const int32_t* __restrict__ uB = p.uid + (int64_t)refB * p.Rp;
            for (int j = lane; j < rA; j += 32) rank_s[j] = (unsigned char)uA[j];
            for (int j = lane; j < rB; j += 32) rank_s[32 * CMAX + j] = (unsigned char)uB[j];
        }
        __syncwarp();
        int mx = 0;
        // the duo's column count: the longer reference decides (warp-uniform), one copy of the
        // two passes per count
        auto run = [&](auto cols) {
            constexpr int C = decltype(cols)::value;
            // ---- the sheet -> bitmaps over distinct tokens, lane = row (32 rows from `first`) ---
            auto convert = [&](const int first) {
                const int i = first + lane;
                if (i > maxsteps) return;
                unsigned bitsA = 0u, bitsB = 0u;
                const unsigned* __restrict__ row = sheet_s + (i & (LEVM_RING - 1)) * LEVM_SHEET_WORDS;
#pragma unroll 4
                for (int k = 0; k < 16; ++k) {
                    unsigned w = row[k];
                    while (w != 0u) {  // (rare: a row has a handful of minimal cells)
                        const int b = 31 - __clz((int)w);
                        w ^= 1u << b;
                        const int l = 2 * k + (b >> 4);        // the lane that set it
                        const int c = C - 1 - (b & 7);         // its cell
                        const int j = l * C + c + 1 - 32 * C;  // column minus r
                        if (b & 8) {
                            const int jj = j + rB;
                            if (jj >= 0 && jj < rB) bitsB |= 1u << rank_s[32 * CMAX + jj];
                        } else {
                            const int jj = j + rA;
                            if (jj >= 0 && jj < rA) bitsA |= 1u << rank_s[jj];
                        }
                    }
                }
                if (i < p.Hout) {
                    if (pairA >= 0 && i <= stepsA) {
                        p.dbits[((int64_t)i * p.P + pairA) * p.Wd] = bitsA;
                        const int cnt = __popc(bitsA);
                        mx = cnt > mx ? cnt : mx;
                    }
                    if (pairB >= 0 && i <= stepsB) {
                        p.dbits[((int64_t)i * p.P + pairB) * p.Wd] = bitsB;
                        const int cnt = __popc(bitsB);
                        mx = cnt > mx ? cnt : mx;
                    }
                }
            };
            auto nothing = [](int) {};
            levm_pass<C, 0>(p, lane, rA, rB, pairA, pairB, maxsteps, nht_s, rowmin_s, sheet_s, nothing);
            __syncwarp();
            levm_pass<C, 1>(p, lane, rA, rB, pairA, pairB, maxsteps, nht_s, rowmin_s, sheet_s, convert);
            __syncwarp();
        };
        const int rmax = rA > rB ? rA : rB;
        const int cneed = (rmax + 32) / 32;  // ceil((r + 1) / 32)
        if (CMAX >= 8 && cneed > 7) run(LevmCols<(CMAX >= 8 ? 8 : CMAX)>{});
        else if (CMAX >= 7 && cneed > 6) run(LevmCols<(CMAX >= 7 ? 7 : CMAX)>{});
        else if (CMAX >= 6 && cneed > 5) run(LevmCols<(CMAX >= 6 ? 6 : CMAX)>{});
        else if (CMAX >= 5 && cneed > 4) run(LevmCols<(CMAX >= 5 ? 5 : CMAX)>{});
        else if (CMAX >= 4 && cneed > 3) run(LevmCols<(CMAX >= 4 ? 4 : CMAX)>{});
        else if (CMAX >= 3 && cneed > 2) run(LevmCols<(CMAX >= 3 ? 3 : CMAX)>{});
        else if (CMAX >= 2 && cneed > 1) run(LevmCols<(CMAX >= 2 ? 2 : CMAX)>{});
        else run(LevmCols<1>{});
        // SM:271-278: prefix 0 points at reference position 0 whenever the reference is non-empty
        if (lane == 0 && p.Hout > 0) {
            if (pairA >= 0 && rA > 0) {
                p.dbits[(int64_t)pairA * p.Wd] = 1u << rank_s[0];
                mx = mx < 1 ? 1 : mx;
            }
            if (pairB >= 0 && rB > 0) {
                p.dbits[(int64_t)pairB * p.Wd] = 1u << rank_s[32 * CMAX];
                mx = mx < 1 ? 1 : mx;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {  // SM:510-511: largest target set -> global maximum U
            const int other = __shfl_xor_sync(LEV_FULL_MASK, mx, o);
            mx = other > mx ? other : mx;
        }
        if (lane == 0 && mx > 0) atomicMax(p.umax, mx);
        __syncwarp();  // the next duo reuses the sheet
    }
}

// Enqueues the packed kernel if the call's shapes and costs admit it; returns 1 then (the caller
// sets LevParams::mask16 for the lev_warp_kernel launch behind it), 0 if not, < 0 on errors.
int lev_launch_mask16(const LevParams& p, bool float_path, cudaStream_t st) {
    // (few pairs: a warp per pair on lev_warp_kernel finishes sooner than half as many warps here)
    int64_t min_pairs = 2048;
    if (const char* e = getenv("B200LEV_MASK16_MIN_PAIRS")) min_pairs = atoll(e);
    if (float_path || p.P < min_pairs || p.P <= 0) return 0;
    const int maxc = p.ins_i > p.del_i ? (p.ins_i > p.sub_i ? p.ins_i : p.sub_i)
                                       : (p.del_i > p.sub_i ? p.del_i : p.sub_i);
    if (p.ins_i < 0 || p.del_i < 0 || p.sub_i < 0 || (int64_t)maxc * (p.R + p.H + 2) >= LEVM_BIG16) return 0;
    if (p.R + 1 > 256) return 0;
    const int C = p.R + 1 <= 64 ? 2 : (p.R + 1 <= 128 ? 4 : 8);
    const int Hs = p.H + 2;
    const size_t per_warp = sizeof(unsigned) * ((size_t)Hs * 2 + LEVM_RING * LEVM_SHEET_WORDS + (2 * 32 * C) / 4);
    const size_t budget = 56 * 1024;  // four CTAs per SM
    if (per_warp > budget) return 0;
    int wpc = (int)(budget / per_warp);
    if (wpc > 4) wpc = 4;  // small CTAs: a batch is often a single wave, and whole CTAs are what the SMs share out
    const size_t smem = per_warp * wpc;
    const int64_t nduo = ((int64_t)p.P + 1) / 2;
    int64_t blocks = (nduo + wpc - 1) / wpc;
    if (blocks > 148 * 32) blocks = 148 * 32;
    auto go = [&](auto kern) -> int {
        if (smem > 48 * 1024 &&
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return lev_check_cuda("cudaFuncSetAttribute");
        lev_launch(kern, dim3((unsigned)blocks), dim3((unsigned)(32 * wpc)), smem, st, p, Hs);
        return B200LEV_OK;
    };
    if (getenv("B200LEV_TRACE"))
        fprintf(stderr, "b200lev: lev_mask16_kernel<%d> P=%d R=%d H=%d warps/CTA=%d smem=%zu\n", C, p.P, p.R, p.H, wpc, smem);
    lev_prof_begin(LEV_PROF_MASK16, st);
    int rc;
    if (C == 2)
        rc = go(lev_mask16_kernel<2>);
    else if (C == 4)
        rc = go(lev_mask16_kernel<4>);
    else
        rc = go(lev_mask16_kernel<8>);
    lev_prof_end(LEV_PROF_MASK16, st);
    if (rc) return rc;
    rc = lev_check_cuda("lev_mask16_kernel");
    return rc ? rc : 1;
}
