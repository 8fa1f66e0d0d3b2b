// lev_bitvec.cuh -- pieces shared by the unit-cost bit-vector kernels (lev_bvfused.cu: Kb, the
// n-best kernel; lev_bvshort.cu: Ks, the short-reference kernel) and their host-side selection
// (lev_bitvec.cu).
#pragma once
#include "lev_common.cuh"

constexpr int LEV_BV_NT = 4;  // tables per warp = runs of identical references per pass

struct LevBvArgs {
    const void* ref;  // raw token tensors, stride 1 along the batch axis
    const void* hyp;
    int64_t ref_st, hyp_st;  // elements between positions
    int R, H, P, ref_group;
    int has_eos;
    int64_t eos;
    int include_eos;
    int32_t* ref_len;  // [Nref]  (same workspace slots K0 fills on the other paths)
    int32_t* hyp_len;  // [P]
    int* counter;      // Kb: the next block of 32 pairs to claim (zeroed by the probe or a memset)
    int32_t* flags;    // caller's warning flags, may be NULL
    int32_t* state;  // workspace state words; [3] != 0 = "not for this path" (lev_bv_took)
    int check_state;   // device-selected mode: veto through state[3] instead of multi-pass
    int slots_log2;    // s: 2^s hash buckets per table, 4 ways each; 2^s > R (positions fit s bits)
    int mode, norm, exclude_last, Hout;
    float mult, padding;
    float* out;
    int64_t out_si;  // prefix: elements between output rows (pairs are adjacent)
    double* acc;     // FINAL, short-reference kernel: += [sum(out), sum(ref_len per pair), #pairs] (may be NULL)
    // b200lev_final_cross through Ks (final mode): pair p reads hypothesis column
    // (p / cross_ab) * cross_b + p % cross_b, cross_ab = A * B and cross_b = B (0: the plain form)
    int cross_ab, cross_b;
};

// Bucketed hash: 4 ways per bucket.  x = v * mult (odd mult: a bijection on 32 bits) picks the
// bucket with its top s bits, and its low 32 - s bits -- the residual -- tell apart every int32
// token of that bucket.  A way holds (x << s) | position, so ONE 128-bit read of the bucket and
// four DPX add-mins settle a look-up (lev_bv_row): no loop, no position side table, and 32 lanes
// with 32 different tokens cost the same as one.  A run leader builds its table with the first
// of a few multipliers under which no bucket overflows (load <= 1 token per bucket on average: a
// couple of tries at most).
// (a build with R = 127 distinct tokens in 128 buckets fails with p = 0.35: 16 tries leave
// 6e-8 of the runs to the slow exact path; R = 128 has 256 buckets, p = 0.04; the typical
// R ~ 100 needs 1.2 tries on average)
constexpr int LEV_BV_TRIES = 16;
__device__ __forceinline__ unsigned lev_bv_mult(int seed) {
    return (0x9E3779B1u * (2u * (unsigned)seed + 1u)) ^ ((unsigned)seed * 0x85EBCA6Au);
}
// A free way holds the all-ones residual and position z = R (the all-zero row of the match
// masks): a token with that residual reads z from it, which is right as long as no real way
// holds it -- and a real way with that residual holds a position < R, which the min prefers.
__device__ __forceinline__ unsigned lev_bv_free_way(int s, int z) { return (~0u << s) | (unsigned)z; }
// The row of a token: nx = -(x << s) (= v * (mult * -2^s), one multiply), z = R < 2^s.  A way's
// key + nx is its position when the residuals agree and >= 2^s otherwise, so the min over the
// four ways and z is the position of the way holding the token, or z.  The table build stops at
// the way this picks, so the build and the look-ups agree on it.
__device__ __forceinline__ unsigned lev_bv_row(const uint4 k, unsigned nx, unsigned z) {
    unsigned u = __viaddmin_u32(k.x, nx, z);
    u = __viaddmin_u32(k.y, nx, u);
    u = __viaddmin_u32(k.z, nx, u);
    return __viaddmin_u32(k.w, nx, u);
}

// Runs of identical references inside a block of 32 consecutive pairs, from each lane's
// "same as the lane before" bit: leader lane of the run, its index, number of runs.
struct LevBvRuns {
    int lead, index, count, len;
    unsigned mask;  // the lanes of my run
};
__device__ __forceinline__ LevBvRuns lev_bv_runs(bool same, int lane) {
    const unsigned starts = ~__ballot_sync(LEV_FULL_MASK, same && lane > 0);
    const unsigned upto = starts & (0xffffffffu >> (31 - lane));
    LevBvRuns r;
    r.lead = 31 - __clz((int)upto);
    r.index = __popc(upto) - 1;
    r.count = __popc(starts);
    const unsigned higher = r.lead == 31 ? 0u : (starts & ~(0xffffffffu >> (31 - r.lead)));
    const int next = higher ? __ffs((int)higher) - 1 : 32;
    r.len = next - r.lead;
    r.mask = (r.len == 32 ? 0xffffffffu : ((1u << r.len) - 1u)) << r.lead;
    return r;
}

// sum = t + pv over W 32-bit words (carry chain in one asm block)
template <int W>
__device__ __forceinline__ void lev_bv_add(const unsigned (&t)[W], const unsigned (&pv)[W],
                                           unsigned (&sum)[W]) {
#ifdef B200LEV_EMU
    unsigned long long carry = 0;
    for (int w = 0; w < W; ++w) {
        const unsigned long long s = (unsigned long long)t[w] + pv[w] + carry;
        sum[w] = (unsigned)s;
        carry = s >> 32;
    }
#else
    if (W == 1) {
        sum[0] = t[0] + pv[0];
    } else if (W == 2) {
        asm("add.cc.u32 %0, %2, %4;\n\taddc.u32 %1, %3, %5;"
            : "=r"(sum[0]), "=r"(sum[W > 1 ? 1 : 0])
            : "r"(t[0]), "r"(t[W > 1 ? 1 : 0]), "r"(pv[0]), "r"(pv[W > 1 ? 1 : 0]));
    } else if (W == 3) {
        asm("add.cc.u32 %0, %3, %6;\n\taddc.cc.u32 %1, %4, %7;\n\taddc.u32 %2, %5, %8;"
            : "=r"(sum[0]), "=r"(sum[W > 1 ? 1 : 0]), "=r"(sum[W > 2 ? 2 : 0])
            : "r"(t[0]), "r"(t[W > 1 ? 1 : 0]), "r"(t[W > 2 ? 2 : 0]), "r"(pv[0]),
              "r"(pv[W > 1 ? 1 : 0]), "r"(pv[W > 2 ? 2 : 0]));
    } else {
        asm("add.cc.u32 %0, %4, %8;\n\taddc.cc.u32 %1, %5, %9;\n\taddc.cc.u32 %2, %6, %10;\n\t"
            "addc.u32 %3, %7, %11;"
            : "=r"(sum[0]), "=r"(sum[W > 1 ? 1 : 0]), "=r"(sum[W > 2 ? 2 : 0]),
              "=r"(sum[W > 3 ? 3 : 0])
            : "r"(t[0]), "r"(t[W > 1 ? 1 : 0]), "r"(t[W > 2 ? 2 : 0]), "r"(t[W > 3 ? 3 : 0]),
              "r"(pv[0]), "r"(pv[W > 1 ? 1 : 0]), "r"(pv[W > 2 ? 2 : 0]), "r"(pv[W > 3 ? 3 : 0]));
    }
#endif
}

// ---------------------------------------------------------------------------------------
// the two kernels' launchers; the hash-table build of Kb
// ---------------------------------------------------------------------------------------
bool lev_bvshort_supports(int elem_bytes, int64_t R);
int lev_bvshort_launch(const LevBvArgs& a, int elem_bytes, cudaStream_t st);
bool lev_bvfused_supports(int elem_bytes);
int lev_bvfused_launch(const LevBvArgs& a, int elem_bytes, cudaStream_t st, void* after_probe);

// The lanes of a run build its hash table together (warp-collective: every lane calls it).
// Lane i of a run of n lanes takes positions i, i + n, ...: it claims a free way of the token's
// bucket with a CAS, and stops early at a way whose residual is the token's (a duplicate).
// Which occurrence ends up representing a token is a race, and does not matter: a position only
// has to be the SAME for every occurrence and for the hypothesis look-ups, which all read the
// finished table.  Positions past the eos may get in too: their rows receive no bits, so matching
// them is no match.  A build whose bucket overflows is retried under the next multiplier.
// Returns 1 if the run has no usable table (tokens outside int32, or LEV_BV_TRIES overflowing
// builds): the caller compares tokens one by one.
template <typename TT>
__device__ __forceinline__ int lev_bv_build_table(const LevBvArgs& a, uint4* keys4, const int nb,
                                                  const TT* __restrict__ rsrc, const int rst,
                                                  const LevBvRuns& runs, const bool active,
                                                  const int tb, const int run_pos, const int exact0,
                                                  const int lane, int* seed_out) {
    constexpr int NT = LEV_BV_NT;
    const int s = a.slots_log2;
    const unsigned efree = lev_bv_free_way(s, a.R);
    int seed = 0;
    int exact = exact0;
    bool need = active && !exact;
#pragma unroll 1
    for (int attempt = 0; attempt < LEV_BV_TRIES; ++attempt) {
        unsigned clear = 0;  // tables (of this pass) being (re)built
#pragma unroll
        for (int t = 0; t < NT; ++t)
            if (__any_sync(LEV_FULL_MASK, need && tb == t)) clear |= 1u << t;
        if (clear == 0) break;
        __syncwarp();
        for (int i = lane; i < nb * NT; i += 32)
            if ((clear >> (i % NT)) & 1u) keys4[i] = make_uint4(efree, efree, efree, efree);
        __syncwarp();
        bool overflow = false;
        if (need) {
            seed = attempt;
            const unsigned hmul = lev_bv_mult(seed);
            const unsigned lim = 1u << s;
            for (int t0 = run_pos; t0 < a.R; t0 += 8 * runs.len) {
                int vv[8];  // 8 of my positions at a time: the loads overlap
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    vv[k] = (t0 + k * runs.len < a.R) ? (int)rsrc[(int64_t)(t0 + k * runs.len) * rst] : 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int t = t0 + k * runs.len;
                    if (t >= a.R) break;
                    const unsigned x = (unsigned)vv[k] * hmul;
                    const unsigned key = (x << s) | (unsigned)t;
                    unsigned* kk = reinterpret_cast<unsigned*>(&keys4[(int)(x >> (32 - s)) * NT + tb]);
                    int w = 0;
                    for (; w < 4; ++w) {
                        const unsigned old = atomicCAS(&kk[w], efree, key);
                        if (old == efree || old - (x << s) < lim) break;  // claimed / the token is there
                    }
                    overflow |= w == 4;
                }
            }
        }
        // the run retries (next multiplier) if any of its lanes met a full bucket
        const bool run_bad = (__ballot_sync(LEV_FULL_MASK, overflow) & runs.mask) != 0;
        need = need && run_bad;
        if (need && attempt == LEV_BV_TRIES - 1) {
            need = false;
            exact = 1;
        }
    }
    __syncwarp();
    *seed_out = seed;
    return exact;
}
