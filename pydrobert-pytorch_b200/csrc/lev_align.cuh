// lev_align.cuh -- b200lev_error_alignment: the walk back along the path b200lev_error_counts
// counts.
//
// Both forms keep, for every DP cell (i >= 1, j >= 1), the predecessor the count cell picks
// (SM:292-314; ties: substitution over insertion over deletion) as a 2-bit field holding the op
// code itself: diagonal with equal tokens 0 (correct), diagonal with different tokens
// 1 (substitution), left 2 (deletion), up 3 (insertion).  The walk therefore reads no token: from
// cell (h, r) it moves to (i-1, j-1) for 0 / 1, (i, j-1) for 2 and (i-1, j) for 3; on row 0 the
// remaining steps are deletions, on column 0 insertions.  It writes the op of the step it takes
// at position k - 1, from r + I - 1 down to 0, and -1 at positions r + I and beyond.
//
// Each form stores the fields in the layout its kernel writes with coalesced stores; an
// addressing policy (code(i, j) -> the 2-bit field of cell (i, j)) reads it back.
//   LevTraceRows   short form (lev_counts.cuh): one lane per pair, rows of RM / 16 words,
//                  [row i-1][word][pair] -- one 128-byte store per word across the warp.
//   LevTraceStrips long form (lev_warp_kernel): C columns per lane in one uint16 (C = 8) or
//                  byte (C = 4), [strip][anti-diagonal step s][lane] per pair, so the 32 lanes
//                  of one step write adjacent slots.
//
// Compiled as part of lev_dp.cu (included at its top).
#pragma once

template <typename A>
__device__ __forceinline__ void lev_align_walk(const A& a, int i, int j, const int len, const int total,
                                               int8_t* __restrict__ out, const int64_t sk) {
    for (int k = len; k < total; ++k) out[(int64_t)k * sk] = (int8_t)-1;
    int64_t at = (int64_t)len * sk;
    while (i > 0 && j > 0) {
        const int op = a.code(i, j);
        at -= sk;
        out[at] = (int8_t)op;
        i -= op != 2;
        j -= op != 3;
    }
    for (; j > 0; --j) {
        at -= sk;
        out[at] = (int8_t)2;
    }
    for (; i > 0; --i) {
        at -= sk;
        out[at] = (int8_t)3;
    }
}

// short form: word w of row i-1 holds columns 16 w + 1 .. 16 w + 16; `base` is the pair's column
struct LevTraceRows {
    const uint32_t* base;
    int64_t row_stride, word_stride;  // NW * P, P
    __device__ __forceinline__ int code(int i, int j) const {
        const uint32_t w = base[(int64_t)(i - 1) * row_stride + (int64_t)((j - 1) >> 4) * word_stride];
        return (int)(w >> (2 * ((j - 1) & 15))) & 3;
    }
};

// long form: the strip geometry of lev_warp_pair (strips of W = 32 C columns, right-aligned so the
// last one ends at column r; lane l of strip k owns columns jb + l C + 1 .. jb + l C + C with
// jb = r - (S - k) W, and updates row i at step s = i + l)
template <int C>
struct LevTraceStrips {
    typedef typename std::conditional<C == 8, uint16_t, uint8_t>::type Field;
    const Field* base;
    int r, S;
    int64_t ns;  // step slots per strip
    __device__ __forceinline__ int code(int i, int j) const {
        constexpr int W = 32 * C;
        const int q = (r - j) / W;               // strips right of j's
        const int off = j - r + (q + 1) * W - 1;  // column within the strip, 0 .. W-1
        const int lane = off / C, c = off % C;
        const Field f = base[((int64_t)(S - 1 - q) * ns + (i + lane - 1)) * 32 + lane];
        return (int)(f >> (2 * c)) & 3;
    }
};

// long form, after lev_warp_kernel<..., TRACE>: one thread per pair
template <int C>
__global__ void __launch_bounds__(256) lev_align_walk_kernel(const LevParams p) {
    typedef typename LevTraceStrips<C>::Field Field;
    for (int64_t pair = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pair < p.P;
         pair += (int64_t)gridDim.x * blockDim.x) {
        const int r = p.ref_len[pair], h = p.hyp_len[pair];
        LevTraceStrips<C> a;
        a.base = reinterpret_cast<const Field*>(p.trace + pair * p.trace_pair_bytes);
        a.r = r;
        a.S = (r + 32 * C) / (32 * C);
        a.ns = p.trace_steps;
        lev_align_walk(a, h, r, r + p.align_ins[pair], p.ops_steps, p.ops + pair * p.ops_sn, p.ops_sk);
    }
}
