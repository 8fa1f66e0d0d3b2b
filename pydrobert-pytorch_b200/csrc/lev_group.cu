// lev_group.cu -- K1s: the throughput kernel for large ragged batches of short/mid pairs.
//
// Same anti-diagonal wavefront as lev_dp.cu, re-shaped so that warps do not idle on
// padding (north star item 3):
//   * a pair is handled by a GROUP of G lanes (G = 2..32, chosen from the padded
//     reference length), each lane owning C adjacent DP columns in registers, so the
//     ramp of the skewed wavefront costs G-1 steps instead of 31 and one __shfl_up_sync
//     serves C cells;
//   * the whole row fits one strip (G*C >= r+1, right-aligned, virtual +BIG columns on
//     the left) -- no shared-memory boundary column;
//   * LENGTH BUCKETS: the batch is counting-sorted on the device by (column class C,
//     hypothesis length) -- histogram built by the packing pass (lev_pack.cu), scan +
//     scatter by lev_sort_kernel -- into a table of TASKS: 32/G pairs (2 x 32/G in the
//     packed path) of the SAME class and near-equal length, largest first.  Warps take
//     tasks round-robin and run their pairs in lock step: lane utilisation is
//     (r+1)/(G*C) instead of (r+1)/(32*C) and no step is spent on a finished pair;
//   * warps are independent (no block barrier anywhere): the task descriptors two tasks
//     ahead and the hypothesis rows one task ahead are already in flight (cp.async /
//     LDGSTS into the other half of a double buffer) while the current task runs;
//   * prefix values are parked in shared memory by the one lane that owns column r and
//     written out after the task by all lanes (scale, IEEE division by the reference
//     length, padding fill: SM:356-386), off the DP loop.
//
// PACKED path: when K0 found all tokens inside a 65536-wide window (their low 16 bits are
// then injective) and costs/lengths keep every value below LEVG_BIG16, TWO pairs share
// each register, one per 16-bit half, and the 2-wide DPX instructions do the work.  Per 2
// cells: VIADDMNMX.U16x2 (token + negated row token, clamped -> 0/1 per half), IMAD (diag +
// neq*sub, FMA pipe), 2 x VIADDMNMX.S16x2.  Otherwise the 32-bit cell update of lev_dp.cu runs.
//
// Integer costs only (cost row, or (cost, count) rows for the error-rate family);
// FINAL and PREFIX modes.  Everything else stays on lev_dp.cu.
#include <cstdlib>

#include "lev_common.cuh"

#define LEVG_NCLS LEV_GROUP_NCLS
// "infinity" of the packed path: BIG16 + (largest reachable value) must stay < 2^15
#define LEVG_BIG16 16000
#ifndef LEVG_MIN_CTAS
#define LEVG_MIN_CTAS 4
#endif

struct LevGroupGeom {
    int G;          // lanes per pair
    int row_words;  // 32-bit words per staged hypothesis row (multiple of 4)
    int allow16;    // costs and lengths admit the packed 2 x int16 DPX path
    int wpc;        // warps per CTA
};

// device-side choice between the packed and the 32-bit build (see lev_pack.cu): lev_tokens_narrow

// IEEE-754 correctly rounded a / b from the correctly rounded reciprocal y = RN(1/b)
// (Markstein): q0 = RN(a*y), r = a - b*q0 (exact in an FMA), q = RN(q0 + r*y).  Valid for
// the operands here (0 <= a < 2^24, 1 <= b < 2^24 - 1, no exponent corner cases) and
// 3 instructions per element once y is hoisted out of the row loop.
__device__ __forceinline__ float levg_div(float a, float b, float y) {
    const float q0 = __fmul_rn(a, y);
    const float r = __fmaf_rn(-b, q0, a);
    return __fmaf_rn(r, y, q0);
}

// ---------------------------------------------------------------------------------------
// 32-bit path: one pair per lane group
// ---------------------------------------------------------------------------------------
template <bool COUNT, int MODE, int C>
__device__ __forceinline__ void levg_run32(const LevParams& p, const int G, const int pair,
                                           const int r, const int h, const int steps,
                                           const int maxsteps, const int* __restrict__ hyp_row) {
    const int lane = threadIdx.x & 31;
    const int gl = lane & (G - 1);
    const int refcol = pair >= 0 ? pair / p.ref_group : 0;
    const int32_t* __restrict__ rtok = p.ref_tok + (int64_t)refcol * p.Rp;
    const int insc = p.ins_i, delc = p.del_i, subc = p.sub_i;
    const int j0 = r - G * C + gl * C + 1;  // right-aligned: the group's last column is r
    int v[C], m[C], rt[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int j = j0 + c;
        v[c] = (j >= 0) ? j * delc : LEV_BIG_I32;  // SM:258-263
        m[c] = j >= 0 ? j : 0;                      // SM:260
        rt[c] = (j >= 1 && pair >= 0) ? rtok[j - 1] : 0;
    }
    (void)m;
    int pl_v = LEV_BIG_I32, pl_m = 0;
    (void)pl_m;
    const bool owner = (gl == G - 1);
    // PREFIX: the lane that owns column r streams the raw row values to the workspace
    // (one 4-byte store per step); lev_prefix_finalize_kernel turns them into the output
    int* __restrict__ raw_row = p.raw32 + (int64_t)(pair >= 0 ? pair : 0) * p.Hr;
    const int nsteps = maxsteps + G - 1;
    for (int s = 1; s <= nsteps; ++s) {
        const int sh_v = __shfl_up_sync(LEV_FULL_MASK, v[C - 1], 1, G);
        const int in_v = (gl == 0) ? LEV_BIG_I32 : sh_v;
        const int diag_v = pl_v;
        pl_v = in_v;
        int in_m = 0, diag_m = 0;
        if (COUNT) {
            const int sh_m = __shfl_up_sync(LEV_FULL_MASK, m[C - 1], 1, G);
            in_m = (gl == 0) ? 0 : sh_m;
            diag_m = pl_m;
            pl_m = in_m;
        }
        (void)in_m; (void)diag_m;
        const int i = s - gl;
        if ((unsigned)(i - 1) < (unsigned)steps) {
            const int ht = hyp_row[i - 1];
            if (COUNT) {  // SM:292-314
                int dc = diag_v, dm = diag_m, lc = in_v, lm = in_m;
                const unsigned nht = 0u - (unsigned)ht;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const int uc = v[c], um = m[c];
                    const int neq = (int)__viaddmin_u32((unsigned)rt[c], nht, 1u);  // 1 = tokens differ (DPX)
                    const int sub_c = dc + neq * subc;
                    const int ins_c = uc + insc;
                    const bool ps = ins_c >= sub_c;
                    int cc = ps ? sub_c : ins_c;
                    int mm = ps ? dm + neq : um + 1;
                    const int del_c = lc + delc;
                    const bool keep = del_c >= cc;
                    cc = keep ? cc : del_c;
                    mm = keep ? mm : lm + 1;
                    dc = uc;
                    dm = um;
                    lc = cc;
                    lm = mm;
                    v[c] = cc;
                    m[c] = mm;
                }
            } else {
                int dg = diag_v, lf = in_v;
                const unsigned nht = 0u - (unsigned)ht;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const int up = v[c];
                    const int sb = dg + (int)(__viaddmin_u32((unsigned)rt[c], nht, 1u) * (unsigned)subc);
                    const int t = __viaddmin_s32(up, insc, sb);
                    lf = __viaddmin_s32(lf, delc, t);
                    dg = up;
                    v[c] = lf;
                }
            }
            if (MODE == LEV_MODE_PREFIX && owner) raw_row[i] = COUNT ? m[C - 1] : v[C - 1];
        }
    }
    if (MODE == LEV_MODE_FINAL && owner && pair >= 0) {  // SM:390-405
        float val = (float)(COUNT ? m[C - 1] : v[C - 1]) * p.mult;
        if (p.norm) val = (r == 0) ? (h > 0 ? 1.0f : 0.0f) : val / (float)r;
        p.out[pair] = val;
    }
}

// ---------------------------------------------------------------------------------------
// packed path: two pairs per lane group, one per 16-bit half.  Both run `maxsteps` rows;
// rows past a pair's own length are never read back.  Cost row only.
// ---------------------------------------------------------------------------------------
template <int MODE, int C>
__device__ __forceinline__ void levg_run16(const LevParams& p, const int G, const int pairA,
                                           const int rA, const int pairB, const int rB,
                                           const int maxsteps,
                                           const unsigned short* __restrict__ hypA,
                                           const unsigned short* __restrict__ hypB,
                                           const int stepsA, const int stepsB,
                                           const int hA, const int hB) {
    const int lane = threadIdx.x & 31;
    const int gl = lane & (G - 1);
    const int32_t* __restrict__ rtA = p.ref_tok + (int64_t)(pairA >= 0 ? pairA / p.ref_group : 0) * p.Rp;
    const int32_t* __restrict__ rtB = p.ref_tok + (int64_t)(pairB >= 0 ? pairB / p.ref_group : 0) * p.Rp;
    const unsigned ins2 = (unsigned)p.ins_i * 0x00010001u, del2 = (unsigned)p.del_i * 0x00010001u;
    const unsigned subc = (unsigned)p.sub_i;
    const unsigned BIG2 = (unsigned)LEVG_BIG16 * 0x00010001u;
    const int j0A = rA - G * C + gl * C + 1, j0B = rB - G * C + gl * C + 1;
    unsigned v[C], rt[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int jA = j0A + c, jB = j0B + c;
        const unsigned vA = (jA >= 0) ? (unsigned)(jA * p.del_i) : (unsigned)LEVG_BIG16;
        const unsigned vB = (jB >= 0) ? (unsigned)(jB * p.del_i) : (unsigned)LEVG_BIG16;
        v[c] = vA | (vB << 16);
        const unsigned tA = (jA >= 1 && pairA >= 0) ? ((unsigned)rtA[jA - 1] & 0xffffu) : 0u;
        const unsigned tB = (jB >= 1 && pairB >= 0) ? ((unsigned)rtB[jB - 1] & 0xffffu) : 0u;
        rt[c] = tA | (tB << 16);
    }
    unsigned pl = BIG2;
    const bool owner = (gl == G - 1);
    unsigned short* __restrict__ rawA = p.raw16 + (int64_t)(pairA >= 0 ? pairA : 0) * p.Hr16;
    unsigned short* __restrict__ rawB = p.raw16 + (int64_t)(pairB >= 0 ? pairB : 0) * p.Hr16;
    const int nsteps = maxsteps + G - 1;
    for (int s = 1; s <= nsteps; ++s) {
        const unsigned sh = __shfl_up_sync(LEV_FULL_MASK, v[C - 1], 1, G);
        const unsigned in = (gl == 0) ? BIG2 : sh;
        unsigned dg = pl;
        pl = in;
        const int i = s - gl;
        if ((unsigned)(i - 1) < (unsigned)maxsteps) {
            // the row's two tokens, NEGATED per half: rt + (-ht) modulo 65 536 is zero where equal,
            // and the DPX add-and-clamp below turns it into the 0 / 1 "differs" in one instruction
            const unsigned htA = hypA[i - 1], htB = hypB[i - 1];
            const unsigned nht = ((0u - htA) & 0xffffu) | ((0u - htB) << 16);
            unsigned lf = in;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const unsigned up = v[c];
                const unsigned n01 = __viaddmin_u16x2(rt[c], nht, 0x00010001u);
                const unsigned sb = n01 * subc + dg;
                const unsigned t = __viaddmin_s16x2(up, ins2, sb);
                lf = __viaddmin_s16x2(lf, del2, t);
                dg = up;
                v[c] = lf;
            }
            if (owner) {
                const unsigned last = v[C - 1];
                if (MODE == LEV_MODE_PREFIX) {
                    // raw row values of both pairs to the workspace (rows past a pair's own
                    // length are never read by the finalize kernel)
                    if (i <= stepsA) rawA[i] = (unsigned short)(last & 0xffffu);
                    if (i <= stepsB) rawB[i] = (unsigned short)(last >> 16);
                } else {
                    // FINAL (SM:390-405): each pair's value is complete at its own last row
                    if (i == stepsA && pairA >= 0) {
                        float val = __fmul_rn((float)(last & 0xffffu), p.mult);
                        if (p.norm) val = (rA == 0) ? (hA > 0 ? 1.0f : 0.0f) : val / (float)rA;
                        p.out[pairA] = val;
                    }
                    if (i == stepsB && pairB >= 0) {
                        float val = __fmul_rn((float)(last >> 16), p.mult);
                        if (p.norm) val = (rB == 0) ? (hB > 0 ? 1.0f : 0.0f) : val / (float)rB;
                        p.out[pairB] = val;
                    }
                }
            }
        }
    }
    if (MODE == LEV_MODE_FINAL && owner) {  // pairs with no hypothesis rows at all
        if (stepsA == 0 && pairA >= 0) {
            float val = __fmul_rn((float)(rA * p.del_i), p.mult);
            if (p.norm) val = (rA == 0) ? (hA > 0 ? 1.0f : 0.0f) : val / (float)rA;
            p.out[pairA] = val;
        }
        if (stepsB == 0 && pairB >= 0) {
            float val = __fmul_rn((float)(rB * p.del_i), p.mult);
            if (p.norm) val = (rB == 0) ? (hB > 0 ? 1.0f : 0.0f) : val / (float)rB;
            p.out[pairB] = val;
        }
    }
}

// ---------------------------------------------------------------------------------------
// bucketing: scan the (class, length) histogram and scatter the pairs into task slots
// ---------------------------------------------------------------------------------------
// what two memsets do on the plain path (cursors + meta := 0, slot table := all ones), as a
// kernel that stands by when the bit-vector kernels took the call
__global__ void __launch_bounds__(256)
lev_group_clear_kernel(const LevParams p, const int64_t ncursor, const int64_t nslots) {
    if (p.bv_check && lev_bv_took(p.wide_flag)) return;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t k = tid; k < ncursor; k += stride) p.gcursor[k] = 0;
    for (int64_t k = tid; k < nslots; k += stride) p.slots[k] = make_int4(-1, -1, -1, -1);
}

#define LEVG_SORT_PER_THREAD 2
__global__ void __launch_bounds__(256)
lev_sort_kernel(const LevParams p, const LevGroupGeom geo, const int count_mode) {
    LEV_DYN_SMEM(int, base);          // [nbins] exclusive offsets of the bins (global)
    int* lhist = base + p.nbins;      // [nbins] this CTA's pairs per bin
    int* goff = lhist + p.nbins;      // [nbins] this CTA's reserved offset inside each bin
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (p.bv_check && lev_bv_took(p.wide_flag)) return;
    if (*p.wide_flag & B200LEV_FLAG_WIDE_TOKENS) return;
    const bool packed = !count_mode && geo.allow16 && lev_tokens_narrow(p.wide_flag);
    const int PPT = (32 / geo.G) * (packed ? 2 : 1);
    const int H1 = p.H + 1;
    // every CTA repeats the (tiny) scan: histogram -> shared memory (all threads), then one
    // warp per class turns it into exclusive offsets, class segments padded to whole tasks
    for (int b = tid; b < p.nbins; b += blockDim.x) {
        base[b] = p.ghist[b];
        lhist[b] = 0;
    }
    __syncthreads();
    // one warp per class segment: exclusive offsets relative to the segment's start; the
    // segment starts (each rounded up to whole tasks) are combined after the barrier
    __shared__ int segtot[LEVG_NCLS];
    if (warp < LEVG_NCLS) {
        const int cseg = warp;
        int carry = 0;
        for (int b0 = 0; b0 < H1; b0 += 32) {
            const int b = b0 + lane;
            const int cnt = b < H1 ? base[cseg * H1 + b] : 0;
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(LEV_FULL_MASK, incl, o);
                if (lane >= o) incl += t;
            }
            if (b < H1) base[cseg * H1 + b] = carry + incl - cnt;
            carry += __shfl_sync(LEV_FULL_MASK, incl, 31);
        }
        if (lane == 0) segtot[cseg] = carry;
    }
    // two-level scatter: rank inside the CTA with shared-memory atomics, then ONE global
    // atomic per (CTA, non-empty bin) reserves the CTA's range -- same-address global
    // atomics serialise in L2, and a bin holds hundreds of pairs
    const int pair0 = blockIdx.x * (256 * LEVG_SORT_PER_THREAD);
    int bin[LEVG_SORT_PER_THREAD], rank[LEVG_SORT_PER_THREAD], rr[LEVG_SORT_PER_THREAD],
        hh[LEVG_SORT_PER_THREAD];
#pragma unroll
    for (int u = 0; u < LEVG_SORT_PER_THREAD; ++u) {
        const int pair = pair0 + u * 256 + tid;
        bin[u] = -1;
        rank[u] = rr[u] = hh[u] = 0;
        if (pair < p.P) {
            rr[u] = p.ref_len[pair / p.ref_group];
            hh[u] = p.hyp_len[pair];
            if (rr[u] == 0 && p.norm && p.flags != nullptr)
                atomicOr(p.flags, B200LEV_FLAG_EMPTY_REF);  // SM:360-366, 397-404
            bin[u] = lev_group_bin(rr[u], hh[u], geo.G, p.H);
        }
    }
    // (the histogram copy above is complete: the scan warp and these atomics touch
    // different arrays, the barrier below orders both against their readers)
#pragma unroll
    for (int u = 0; u < LEVG_SORT_PER_THREAD; ++u)
        if (bin[u] >= 0) rank[u] = atomicAdd(&lhist[bin[u]], 1);
    __syncthreads();
    // all reservations of a thread are issued before the first result is needed
    {
        int got[4], bb[4];
        for (int b0 = tid; b0 < p.nbins; b0 += 4 * blockDim.x) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int b = b0 + k * blockDim.x;
                bb[k] = b;
                got[k] = 0;
                if (b < p.nbins && lhist[b] > 0) got[k] = atomicAdd(&p.gcursor[b], lhist[b]);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (bb[k] < p.nbins) goff[bb[k]] = got[k];
        }
    }
    int segstart[LEVG_NCLS];
    {
        int start = 0;
#pragma unroll
        for (int c = 0; c < LEVG_NCLS; ++c) {
            segstart[c] = start;
            start = (start + segtot[c] + PPT - 1) / PPT * PPT;
        }
        if (blockIdx.x == 0 && tid == 0) p.gmeta[0] = start / PPT;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < LEVG_SORT_PER_THREAD; ++u) {
        if (bin[u] < 0) continue;
        const int cls = lev_group_class(rr[u], geo.G);
        int sstart = 0;
#pragma unroll
        for (int c = 0; c < LEVG_NCLS; ++c)
            if (c == LEVG_NCLS - 1 - cls) sstart = segstart[c];
        const int pos = sstart + base[bin[u]] + goff[bin[u]] + rank[u];
        p.slots[pos] = make_int4(pair0 + u * 256 + tid, rr[u], hh[u], cls);
    }
}

// ---------------------------------------------------------------------------------------
// the DP kernel: independent warps, tasks round-robin, two-deep prefetch
// ---------------------------------------------------------------------------------------
template <bool COUNT, int MODE, bool PACKED>
__global__ void __launch_bounds__(128, LEVG_MIN_CTAS) lev_group_kernel(const LevParams p, const LevGroupGeom geo) {
    LEV_DYN_SMEM(int, smem);
    // Which of the two builds of this kernel runs is decided on the device from what K0
    // found in the tokens (no host round trip): wider than int32 -> neither (the 64-bit
    // compare path of lev_warp_kernel, enqueued right behind, takes the batch); inside a
    // 65536-wide window and small values -> PACKED; else the 32-bit build.
    if (p.bv_check && lev_bv_took(p.wide_flag)) return;
    if (*p.wide_flag & B200LEV_FLAG_WIDE_TOKENS) return;
    if ((!COUNT && geo.allow16 && lev_tokens_narrow(p.wide_flag)) != PACKED) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int G = geo.G, PPW = 32 / G, RW = geo.row_words;
    const int PPT = PACKED ? 2 * PPW : PPW;  // pairs per task (<= 32)
    int* stage_w = smem + (size_t)warp * (2 * PPT * RW);  // [2][PPT][RW]  hypothesis rows
    const int ntasks = p.gmeta[0];
    const int nW = gridDim.x * geo.wpc;
    const int g = lane / G;
    const int CPR = RW / 4;  // 16-byte chunks per staged row
    const int stage_iters = (PPT * CPR + 31) / 32;

    auto load_slot = [&](int t) {
        int4 s = make_int4(-1, 0, 0, 0);
        if (t < ntasks && lane < PPT) s = p.slots[(int64_t)t * PPT + lane];
        if (s.x < 0) s = make_int4(-1, 0, 0, s.w < 0 ? 0 : s.w);
        return s;
    };
    auto stage = [&](const int4& S, int buf) {
        char* dst0 = reinterpret_cast<char*>(stage_w + buf * PPT * RW);
        for (int it = 0; it < stage_iters; ++it) {
            const int c = it * 32 + lane;
            const int k = min(c / CPR, PPT - 1), ch = c - (c / CPR) * CPR;
            const int pk = __shfl_sync(LEV_FULL_MASK, S.x, k);
            const int hk = __shfl_sync(LEV_FULL_MASK, S.z, k);
            const int sk = p.exclude_last ? (hk > 0 ? hk - 1 : 0) : hk;
            if (c < PPT * CPR && pk >= 0 && ch * 16 < sk * (PACKED ? 2 : 4)) {
                const char* src = PACKED
                    ? reinterpret_cast<const char*>(p.hyp_tok16 + (int64_t)pk * p.Hp16)
                    : reinterpret_cast<const char*>(p.hyp_tok + (int64_t)pk * p.Hp);
                lev_cp_async16(dst0 + (size_t)k * RW * 4 + ch * 16, src + ch * 16);
            }
        }
    };

    int t = blockIdx.x * geo.wpc + warp;
    int4 S_cur = load_slot(t), S_nxt = load_slot(t + nW);
    int buf = 0;
    if (t < ntasks) stage(S_cur, buf);
    lev_cp_async_commit();
    while (t < ntasks) {
        if (t + nW < ntasks) stage(S_nxt, buf ^ 1);
        lev_cp_async_commit();
        const int4 S_nn = load_slot(t + 2 * nW);
        lev_cp_async_wait<1>();  // everything but the newest group: this task's rows landed
        __syncwarp();
        const int cls = __shfl_sync(LEV_FULL_MASK, S_cur.w, 0);  // tasks are class-pure
        const int* rows = stage_w + buf * PPT * RW;
        int maxsteps = p.exclude_last ? (S_cur.z > 0 ? S_cur.z - 1 : 0) : S_cur.z;  // SM:286-288
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const int other = __shfl_xor_sync(LEV_FULL_MASK, maxsteps, o);
            maxsteps = other > maxsteps ? other : maxsteps;
        }
        if (PACKED) {
            // group g runs slots 2g (low halves) and 2g+1 (high halves) of the task
            const int pA = __shfl_sync(LEV_FULL_MASK, S_cur.x, 2 * g);
            const int rA = __shfl_sync(LEV_FULL_MASK, S_cur.y, 2 * g);
            const int hA = __shfl_sync(LEV_FULL_MASK, S_cur.z, 2 * g);
            const int pB = __shfl_sync(LEV_FULL_MASK, S_cur.x, 2 * g + 1);
            const int rB = __shfl_sync(LEV_FULL_MASK, S_cur.y, 2 * g + 1);
            const int hB = __shfl_sync(LEV_FULL_MASK, S_cur.z, 2 * g + 1);
            const int sA = p.exclude_last ? (hA > 0 ? hA - 1 : 0) : hA;
            const int sB = p.exclude_last ? (hB > 0 ? hB - 1 : 0) : hB;
            const unsigned short* hA_row = reinterpret_cast<const unsigned short*>(rows + (2 * g) * RW);
            const unsigned short* hB_row = reinterpret_cast<const unsigned short*>(rows + (2 * g + 1) * RW);
#define LEVG_R16(C_) levg_run16<MODE, C_>(p, G, pA, rA, pB, rB, maxsteps, hA_row, hB_row, sA, sB, hA, hB)
            switch (cls) {
                case 0: LEVG_R16(8); break;
                case 1: LEVG_R16(12); break;
                case 2: LEVG_R16(16); break;
                case 3: LEVG_R16(20); break;
                case 4: LEVG_R16(24); break;
                default: LEVG_R16(28); break;
            }
#undef LEVG_R16
        } else {
            const int pair = __shfl_sync(LEV_FULL_MASK, S_cur.x, g);
            const int r = __shfl_sync(LEV_FULL_MASK, S_cur.y, g);
            const int h = __shfl_sync(LEV_FULL_MASK, S_cur.z, g);
            const int steps = p.exclude_last ? (h > 0 ? h - 1 : 0) : h;
            const int* hyp_row = rows + g * RW;
#define LEVG_R32(C_) levg_run32<COUNT, MODE, C_>(p, G, pair, r, h, steps, maxsteps, hyp_row)
            switch (cls) {
                case 0: LEVG_R32(8); break;
                case 1: LEVG_R32(12); break;
                case 2: LEVG_R32(16); break;
                case 3: LEVG_R32(20); break;
                case 4: LEVG_R32(24); break;
                default: LEVG_R32(28); break;
            }
#undef LEVG_R32
        }
        __syncwarp();
        S_cur = S_nxt;
        S_nxt = S_nn;
        t += nW;
        buf ^= 1;
    }
    lev_cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------
// PREFIX epilogue: raw row values -> the caller's (H', N) / (N, H') fp32 tensor.
//   row 0 = r * (1 | del) (SM:279-285); rows 1..steps = raw (SM:340-346); x mult, / r with
//   the empty-reference rule (SM:356-378); rows >= h + (0|1) = padding (SM:379-386).
// Sequence-first output (unit stride along n): 32 rows x 128 pairs tiles are transposed
// through shared memory so that both the raw reads (along rows) and the output writes
// (along pairs, one float4 = 128 bits per thread) are coalesced.
// ---------------------------------------------------------------------------------------
template <bool COUNT>
__device__ __forceinline__ float levg_finalize_one(const LevParams& p, bool packed, int n, int i,
                                                   int r, int h, float y) {
    const int first_pad = h + (p.exclude_last ? 0 : 1);
    if (i >= first_pad) return p.padding;
    int raw;
    if (i == 0)
        raw = COUNT ? r : r * p.del_i;
    else
        raw = packed ? (int)p.raw16[(int64_t)n * p.Hr16 + i] : p.raw32[(int64_t)n * p.Hr + i];
    float val = __fmul_rn((float)raw, p.mult);
    if (p.norm) val = (r == 0) ? (i > 0 ? 1.0f : 0.0f) : levg_div(val, (float)r, y);
    return val;
}

template <bool COUNT>
__global__ void __launch_bounds__(256)
lev_prefix_finalize_kernel(const LevParams p, const LevGroupGeom geo) {
    if (p.bv_check && lev_bv_took(p.wide_flag)) return;
    if (*p.wide_flag & B200LEV_FLAG_WIDE_TOKENS) return;  // lev_warp_kernel wrote `out` itself
    const bool packed = !COUNT && geo.allow16 && lev_tokens_narrow(p.wide_flag);
    const int tid = threadIdx.x;
    if (p.out_sn == 1) {
        // lane = pair: a lane walks 32 rows of ITS pair's raw values (128-bit loads, the row's
        // line stays in L1) and every store instruction writes 32 neighbouring pairs of one
        // output row -- 128 contiguous bytes -- so nothing has to be transposed
        // (work item = 256 pairs x 32 rows; a CTA takes several, which keeps the grid -- and the
        // cost of standing by for the bit-vector path -- small)
        const int segs = (p.Hout + 31) / 32;
        const int64_t items = (int64_t)((p.P + 255) / 256) * segs;
        for (int64_t item = blockIdx.x; item < items; item += gridDim.x) {
        const int n = (int)(item / segs) * 256 + tid;
        const int i0 = (int)(item % segs) * 32;
        if (n >= p.P) continue;
        const int i1 = i0 + 32 < p.Hout ? i0 + 32 : p.Hout;
        const int r = p.ref_len[n / p.ref_group], h = p.hyp_len[n];
        const float rf = (float)r;
        const float y = r > 0 ? __frcp_rn(rf) : 0.0f;
        const int first_pad = h + (p.exclude_last ? 0 : 1);
        const bool norm = p.norm != 0;
        float* __restrict__ o = p.out + (int64_t)i0 * p.out_si + n;
        // all four 128-bit loads of the packed rows are issued before the first value is used
        uint4 w16[4];
        if (packed) {
            const uint4* src = reinterpret_cast<const uint4*>(p.raw16 + (int64_t)n * p.Hr16 + i0);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                w16[k] = (i0 + 8 * k < i1) ? src[k] : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int ib = i0 + 8 * k;
            if (ib >= i1) break;
            int raw[8];
            if (packed) {
                const uint4 w = w16[k];
                raw[0] = (int)(w.x & 0xffffu); raw[1] = (int)(w.x >> 16);
                raw[2] = (int)(w.y & 0xffffu); raw[3] = (int)(w.y >> 16);
                raw[4] = (int)(w.z & 0xffffu); raw[5] = (int)(w.z >> 16);
                raw[6] = (int)(w.w & 0xffffu); raw[7] = (int)(w.w >> 16);
            } else {
                const int4* src = reinterpret_cast<const int4*>(p.raw32 + (int64_t)n * p.Hr + ib);
                const int4 w0 = src[0];
                const int4 w1 = ib + 4 < p.Hr ? src[1] : make_int4(0, 0, 0, 0);
                raw[0] = w0.x; raw[1] = w0.y; raw[2] = w0.z; raw[3] = w0.w;
                raw[4] = w1.x; raw[5] = w1.y; raw[6] = w1.z; raw[7] = w1.w;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int i = ib + u;
                if (i < i1) {
                    const int rv = (i == 0) ? (COUNT ? r : r * p.del_i) : raw[u];
                    float val = __fmul_rn((float)rv, p.mult);
                    if (norm) val = (r == 0) ? (i > 0 ? 1.0f : 0.0f) : levg_div(val, rf, y);
                    *o = (i < first_pad) ? val : p.padding;
                    o += p.out_si;
                }
            }
        }
        }
    } else {
        // batch-first (or arbitrary strides): rows of one pair are adjacent in the output
        const int64_t total = (int64_t)p.P * p.Hout;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + tid; e < total;
             e += (int64_t)gridDim.x * blockDim.x) {
            const int n = (int)(e / p.Hout), i = (int)(e - (int64_t)n * p.Hout);
            const int r = p.ref_len[n / p.ref_group], h = p.hyp_len[n];
            const float y = r > 0 ? __frcp_rn((float)r) : 0.0f;
            p.out[(int64_t)i * p.out_si + (int64_t)n * p.out_sn] =
                levg_finalize_one<COUNT>(p, packed, n, i, r, h, y);
        }
    }
}

// geometry + shared-memory footprint of one build
static size_t levg_geometry(const LevParams& p, bool packed, LevGroupGeom* geo) {
    const int PPW = 32 / geo->G, PPT = packed ? 2 * PPW : PPW;
    // staged hypothesis rows: uint16 (packed) or int32; whole 16-byte chunks per row
    geo->row_words = packed ? (int)((p.H + 7) / 8) * 4 : (int)((p.H + 3) / 4) * 4;
    if (geo->row_words < 4) geo->row_words = 4;
    geo->wpc = 4;
    const size_t per_warp = sizeof(int) * ((size_t)2 * PPT * geo->row_words);
    return per_warp * geo->wpc;
}

template <bool COUNT, int MODE, bool PACKED>
static int levg_launch_one(const LevParams& p, LevGroupGeom geo, cudaStream_t st) {
    const size_t smem = levg_geometry(p, PACKED, &geo);
    auto kern = lev_group_kernel<COUNT, MODE, PACKED>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            lev_set_error("cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
            return B200LEV_ERR_CUDA;
        }
    }
    // persistent: as many CTAs as stay resident (LEVG_MIN_CTAS per SM by registers, fewer by smem)
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm > LEVG_MIN_CTAS) per_sm = LEVG_MIN_CTAS;
    if (per_sm < 1) per_sm = 1;
    int64_t blocks = 148 * per_sm;
    const int PPT = (32 / geo.G) * (PACKED ? 2 : 1);
    const int64_t max_tasks = (p.P + PPT - 1) / PPT + LEVG_NCLS;
    if (blocks * geo.wpc > max_tasks) blocks = (max_tasks + geo.wpc - 1) / geo.wpc;
    lev_launch(kern, dim3((unsigned)blocks), dim3(32 * geo.wpc), smem, st, p, geo);
    const int rc = lev_check_cuda("lev_group_kernel");
    return rc ? rc : 1;
}

int lev_group_eligible(int64_t R, int64_t H, int64_t P) {
    // small batches: latency matters, one warp per pair (B200LEV_GROUP_MIN_PAIRS
    // overrides the switch-over point; tests use it to drive both kernels)
    int64_t min_pairs = 4096;
    if (const char* e = getenv("B200LEV_GROUP_MIN_PAIRS")) min_pairs = atoll(e);
    if (P < min_pairs || H > 1000 || R > 30000) return 0;
    return lev_group_lanes(R);
}

// Returns 1 if the group kernels took the job, 0 if they do not apply (caller falls back
// to the warp-per-pair kernel), < 0 on error.
int lev_launch_group(const LevParams& p, int mode, bool count_mode, cudaStream_t st) {
    if (mode == LEV_MODE_MASK) return 0;
    LevGroupGeom geo;
    memset(&geo, 0, sizeof(geo));
    geo.G = lev_group_eligible(p.R, p.H, p.P);
    if (geo.G == 0) return 0;
    const int maxc = p.ins_i > p.del_i ? (p.ins_i > p.sub_i ? p.ins_i : p.sub_i)
                                       : (p.del_i > p.sub_i ? p.del_i : p.sub_i);
    geo.allow16 = (!count_mode && p.ins_i >= 0 && p.del_i >= 0 && p.sub_i >= 0 &&
                   (int64_t)maxc * (p.R + p.H + 2) < LEVG_BIG16)
                      ? 1
                      : 0;
    LevGroupGeom tmp = geo;
    if (levg_geometry(p, false, &tmp) > 200 * 1024) return 0;
    tmp = geo;
    if (geo.allow16 && levg_geometry(p, true, &tmp) > 200 * 1024) geo.allow16 = 0;
    // bucketing: clear the scatter cursors + meta and the slot table, then scan + scatter
    if (p.bv_check) {
        // stand-by mode: the clearing stands by as well, so a batch the bit-vector kernel took
        // costs no memsets here
        lev_launch(lev_group_clear_kernel, dim3(148 * 2), dim3(256), 0, st, p,
                   (int64_t)(p.nbins + 16), (int64_t)(p.P + LEVG_NCLS * 32));
    } else if (cudaMemsetAsync(p.gcursor, 0, sizeof(int) * (size_t)(p.nbins + 16), st) != cudaSuccess ||
               cudaMemsetAsync(p.slots, 0xff, 16 * (size_t)(p.P + LEVG_NCLS * 32), st) != cudaSuccess)
        return lev_check_cuda("memset");
    lev_prof_begin(LEV_PROF_SORT, st);
    {
        const int per_cta = 256 * LEVG_SORT_PER_THREAD;
        const size_t sort_smem = 3 * sizeof(int) * (size_t)p.nbins;
        if (sort_smem > 48 * 1024)
            cudaFuncSetAttribute(lev_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)sort_smem);
        lev_launch(lev_sort_kernel, dim3((unsigned)((p.P + per_cta - 1) / per_cta)), dim3(256),
                   sort_smem, st, p, geo, (int)count_mode);
    }
    lev_prof_end(LEV_PROF_SORT, st);
    int rc = lev_check_cuda("lev_sort_kernel");
    if (rc) return rc;
    lev_prof_begin(LEV_PROF_DP, st);
    // both builds are enqueued; the device-side token range decides which one works
#define LEVG_BOTH(COUNT_, MODE_)                                                   \
    rc = levg_launch_one<COUNT_, MODE_, false>(p, geo, st);                        \
    if (rc <= 0) return rc < 0 ? rc : B200LEV_ERR_UNSUPPORTED;                     \
    if (!COUNT_ && geo.allow16) {                                                  \
        rc = levg_launch_one<COUNT_, MODE_, true>(p, geo, st);                     \
        if (rc <= 0) return rc < 0 ? rc : B200LEV_ERR_UNSUPPORTED;                 \
    }
    if (!count_mode) {
        if (mode == LEV_MODE_FINAL) { LEVG_BOTH(false, LEV_MODE_FINAL) }
        else { LEVG_BOTH(false, LEV_MODE_PREFIX) }
    } else {
        if (mode == LEV_MODE_FINAL) { LEVG_BOTH(true, LEV_MODE_FINAL) }
        else { LEVG_BOTH(true, LEV_MODE_PREFIX) }
    }
#undef LEVG_BOTH
    lev_prof_end(LEV_PROF_DP, st);
    if (mode == LEV_MODE_PREFIX && p.Hout > 0) {
        lev_prof_begin(LEV_PROF_FINALIZE, st);
        dim3 grid, block(256);
        if (p.out_sn == 1) {
            int64_t items = (int64_t)((p.P + 255) / 256) * ((p.Hout + 31) / 32);
            if (p.bv_check && items > 148 * 4) {  // stand-by duty: a small grid exits faster
                const int64_t per_cta = (items + 148 * 4 - 1) / (148 * 4);
                items = (items + per_cta - 1) / per_cta;
            }
            grid = dim3((unsigned)items);
        }
        else
            grid = dim3((unsigned)min((int64_t)148 * 16, ((int64_t)p.P * p.Hout + 255) / 256));
        if (count_mode)
            lev_launch(lev_prefix_finalize_kernel<true>, grid, block, 0, st, p, geo);
        else
            lev_launch(lev_prefix_finalize_kernel<false>, grid, block, 0, st, p, geo);
        lev_prof_end(LEV_PROF_FINALIZE, st);
        rc = lev_check_cuda("lev_prefix_finalize_kernel");
        if (rc) return rc;
    }
    return 1;
}
