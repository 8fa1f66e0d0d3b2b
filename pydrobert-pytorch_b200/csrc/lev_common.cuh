// lev_common.cuh -- shared declarations for the Levenshtein kernels.
//
// "SM" in comments is src/pydrobert/torch/_string.py of the reference.
#pragma once
#include "simt.h"

#include "../../include/b200lev.h"

// INFIX: b200lev_infix's distance-only form on the short bit-vector kernel (lev_bvshort.cu)
enum LevMode { LEV_MODE_FINAL = 0, LEV_MODE_PREFIX = 1, LEV_MODE_MASK = 2, LEV_MODE_INFIX = 3 };

// "Infinity" for the int32 DP: virtual columns left of column 0 hold it so that
// column 0 needs no special case.  Costs are bounded on the host so that BIG plus
// any reachable path cost stays below 2^31.
#define LEV_BIG_I32 (1 << 29)

static inline int64_t lev_round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// ---- group kernel bucketing (lev_group.cu, histogram built by lev_pack.cu) ----
#define LEV_GROUP_NCLS 6  // column classes C = 8, 12, ..., 28 per lane
// lanes per pair for a padded reference length R: smallest power of two >= 2 with
// G * 28 >= R + 1; 0 if the group kernel does not apply
static inline int lev_group_lanes(int64_t R) {
    int G = 2;
    while (G <= 32 && (int64_t)G * 28 < R + 1) G <<= 1;
    return G <= 32 ? G : 0;
}
// smallest class whose strip of G*C columns covers columns 0..r
__host__ __device__ static inline int lev_group_class(int r, int G) {
    const int need = (r + G) / G;  // ceil((r + 1) / G)
    const int cls = (need - 8 + 3) >> 2;
    return cls < 0 ? 0 : cls;
}
// histogram bin of a pair: classes descending, then hypothesis lengths descending
__host__ __device__ static inline int lev_group_bin(int r, int h, int G, int H) {
    return (LEV_GROUP_NCLS - 1 - lev_group_class(r, G)) * (H + 1) + (H - h);
}

// b200lev_error_counts / b200lev_error_alignment: the short form (lev_counts.cuh, one lane per
// pair from the raw tokens) takes references up to 64 tokens of the hypotheses' width; the long
// form (K0 + lev_warp_kernel) everything else
static inline bool lev_counts_short_form(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp) {
    return ref->T <= 64 && ref->elem_bytes == hyp->elem_bytes;
}

// b200lev_error_alignment, long form: lev_warp_kernel's fixed strip widths (C columns per lane:
// one uint16 of 2-bit choices for int32 cells, one byte for fp32 cells) and the trace bytes of
// one pair, [strip][anti-diagonal step][lane] with H + 31 steps per strip
#define LEV_ALIGN_C_INT 8
#define LEV_ALIGN_C_FLT 4
static inline int64_t lev_align_pair_bytes(int64_t R, int64_t H, int C) {
    const int64_t W = 32 * C;
    return (R + W) / W * (H + 31) * 32 * (C / 4);
}

// Workspace layout (device scratch supplied by the caller).  All offsets are
// multiples of 128 bytes.
struct LevLayout {
    int64_t R, H, Nref, P;
    int64_t Rp, Hp;  // padded row lengths of the packed int32 token tables
    int64_t Hp16;    // padded row length of the 16-bit hypothesis table (multiple of 8)
    int64_t Hout;    // output rows of the prefix / mask modes
    int64_t Wd;      // 32-bit words of one (prefix, pair) distinct-token bitmap
    size_t off_ref_tok, off_hyp_tok, off_hyp_tok16, off_ref_len, off_hyp_len, off_flags;
    // group kernel (lev_group.cu): [ghist nbins][gcursor nbins][gmeta 16] follow the 4 state
    // words directly (one memset clears state + ghist); slots = sorted task table
    int64_t nbins;
    size_t off_ghist, off_gcursor, off_gmeta, off_slots;
    // raw prefix rows written by the group kernel, read by lev_prefix_finalize_kernel
    int64_t Hr, Hr16;
    size_t off_raw;
    size_t off_uid, off_dtok, off_ndist, off_dbits;
    // bit-vector path (lev_bitvec.cu; final and prefix modes, R <= 128): Kb's block counter
    size_t off_bv_counter;
    // pack kernel, few long sequences: [N first-eos words][ceil(N / 32) tickets] per side
    size_t off_split_ref, off_split_hyp;
    // error alignment (kind 3): the cells' 2-bit choices -- short form [row][word][pair], long
    // form trace_pair_bytes per pair -- and, long form, the insertion count of each pair
    size_t off_trace, off_align_ins;
    int64_t trace_pair_bytes;
    size_t bytes;
};

// kind: 0 = final value, 1 = completion (mask mode), 2 = prefix table, 3 = error alignment
static inline LevLayout lev_layout(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                   int kind, int exclude_last) {
    const int for_completion = (kind == 1);
    LevLayout L;
    L.R = ref->T;
    L.H = hyp->T;
    L.Nref = ref->N;
    L.P = hyp->N;
    L.Rp = lev_round_up(L.R > 0 ? L.R : 1, 4);
    L.Hp = lev_round_up(L.H > 0 ? L.H : 1, 4);
    L.Hp16 = lev_round_up(L.H > 0 ? L.H : 1, 8);
    L.Hout = L.H + (exclude_last ? 0 : 1);
    if (for_completion && L.Hout < 1) L.Hout = 1;  // SM:271-278
    L.Wd = (L.R + 31) / 32;
    if (L.Wd < 1) L.Wd = 1;
    size_t o = 0;
    auto take = [&](size_t n) {
        size_t at = o;
        o += (size_t)lev_round_up((int64_t)n, 128);
        return at;
    };
    L.off_ref_tok = take(sizeof(int32_t) * (size_t)L.Nref * L.Rp);
    L.off_hyp_tok = take(sizeof(int32_t) * (size_t)L.P * L.Hp);
    L.off_hyp_tok16 = take(sizeof(uint16_t) * (size_t)L.P * L.Hp16);
    L.off_ref_len = take(sizeof(int32_t) * (size_t)L.Nref);
    L.off_hyp_len = take(sizeof(int32_t) * (size_t)L.P);
    L.nbins = LEV_GROUP_NCLS * (L.H + 1);
    L.off_flags = take(sizeof(int32_t) * (size_t)(4 + 2 * L.nbins + 16));  // state + group tables
    L.off_ghist = L.off_flags + 4 * sizeof(int32_t);
    L.off_gcursor = L.off_ghist + sizeof(int32_t) * (size_t)L.nbins;
    L.off_gmeta = L.off_gcursor + sizeof(int32_t) * (size_t)L.nbins;
    L.off_slots = take(16 * (size_t)(L.P + LEV_GROUP_NCLS * 32));
    L.Hr = lev_round_up(L.H + 1, 4);
    L.Hr16 = lev_round_up(L.H + 1, 8);
    L.off_raw = (kind == 2) ? take(sizeof(int32_t) * (size_t)L.P * L.Hr) : 0;
    L.off_bv_counter = (kind != 1 && L.R <= 128) ? take(sizeof(int32_t)) : 0;
    L.off_uid = L.off_dtok = L.off_ndist = L.off_dbits = 0;
    if (for_completion) {
        L.off_uid = take(sizeof(int32_t) * (size_t)L.Nref * L.Rp);
        L.off_dtok = take(sizeof(int64_t) * (size_t)L.Nref * L.Rp);
        L.off_ndist = take(sizeof(int32_t) * (size_t)L.Nref);
        L.off_dbits = take(sizeof(uint32_t) * (size_t)L.Hout * L.P * L.Wd);
    }
    L.off_split_ref = take(sizeof(int32_t) * (size_t)(L.Nref + (L.Nref + 31) / 32));
    L.off_split_hyp = take(sizeof(int32_t) * (size_t)(L.P + (L.P + 31) / 32));
    L.off_trace = L.off_align_ins = 0;
    L.trace_pair_bytes = 0;
    if (kind == B200LEV_WS_ALIGN) {
        if (lev_counts_short_form(ref, hyp)) {
            L.off_trace = take(sizeof(uint32_t) * (size_t)(L.R <= 32 ? 2 : 4) * L.H * L.P);
        } else {
            const int64_t bi = lev_align_pair_bytes(L.R, L.H, LEV_ALIGN_C_INT);
            const int64_t bf = lev_align_pair_bytes(L.R, L.H, LEV_ALIGN_C_FLT);
            L.trace_pair_bytes = bi > bf ? bi : bf;
            L.off_trace = take((size_t)L.trace_pair_bytes * L.P);
            L.off_align_ins = take(sizeof(int32_t) * (size_t)L.P);
        }
    }
    L.bytes = o;
    return L;
}

// Everything the DP kernels need, by value.
struct LevParams {
    const int32_t* ref_tok;  // [Nref][Rp]
    const int32_t* hyp_tok;  // [P][Hp]
    const uint16_t* hyp_tok16;  // [P][Hp16] low 16 bits of every hypothesis token
    int64_t Hp16;
    const int32_t* ref_len;  // [Nref]
    const int32_t* hyp_len;  // [P]
    int64_t Rp, Hp;
    int R, H, P, ref_group;
    // costs: integer path uses the *_i fields, float path the *_f fields
    int ins_i, del_i, sub_i;
    float ins_f, del_f, sub_f;
    float mult;  // SM:168-174
    int norm, exclude_last;
    float padding;
    // FINAL: out[n];  PREFIX: out[i*out_si + n*out_sn]
    float* out;
    int64_t out_si, out_sn;
    int Hout;
    // MASK
    const int32_t* uid;  // [Nref][Rp] rank of ref[j] among the pair's distinct tokens
    const int32_t* ndist;  // [Nref] number of distinct tokens of the reference
    uint32_t* dbits;     // [Hout][P][Wd]
    int Wd;
    int* umax;
    int* flags;            // caller's warning flags (may be NULL)
    const int* wide_flag;  // never NULL: workspace state words K0 fills: [0] flags (incl.
                           // B200LEV_FLAG_WIDE_TOKENS), [1], [2] biased token range
    // the caller's tensors, for the 64-bit compare path only
    const void* ref_raw;
    const void* hyp_raw;
    int64_t ref_st, ref_sn, hyp_st, hyp_sn;
    int ref_eb, hyp_eb;
    int only_if_wide;  // lev_warp_kernel: exit unless the wide-token flag is set
    int mask16;        // MASK: lev_mask16_kernel ran first; lev_warp_kernel skips the pairs it took
    int bv_check;      // the bit-vector kernels ran first: exit if they took the batch
    // group kernel tables (workspace)
    int* ghist;
    int* gcursor;
    int* gmeta;   // [0] = number of tasks
    int4* slots;  // sorted (pair, r, h, class) per task slot; pair < 0 = padding
    int* gmeta_order;  // same storage viewed as int[P]: pair order of the CTA kernel
    int32_t* raw32;          // [P][Hr]   raw prefix rows (32-bit group path)
    unsigned short* raw16;   // [P][Hr16] same storage, packed path
    int64_t Hr, Hr16;
    int nbins;
    // b200lev_error_alignment: the cells' choices (short form [row][word][pair] words; long form
    // trace_pair_bytes per pair, trace_steps step slots per strip), the insertions of each pair
    // (long form), and the int8 ops the walk writes, step k of pair n at ops[k*ops_sk + n*ops_sn],
    // k < ops_steps
    unsigned char* trace;
    int64_t trace_pair_bytes, trace_steps;
    int* align_ins;
    int8_t* ops;
    int64_t ops_sk, ops_sn;
    int ops_steps;
    // b200lev_error_counts: (C, S, D, I) of pair n at counts[4n .. 4n+3]
    int64_t* counts;
    // b200lev_infix with spans: the start and end rows of pair n's match
    int64_t* infix_start;
    int64_t* infix_end;
};


#if defined(__CUDACC__) || defined(B200LEV_EMU)
// K0's token range (state[1] = max(u), state[2] = max(~u), u = token + 2^31): all tokens of the
// call lie in one 65 536-wide window, so their low 16 bits tell them apart
__device__ __forceinline__ bool lev_tokens_narrow(const int* state) {
    const unsigned umax = (unsigned)state[1], umin = ~(unsigned)state[2];
    return umax < umin || umax - umin < 65536u;
}
// Mask mode, small alphabets (character-level targets): when every token of the call lies in a
// window of 32 values, "token - smallest token" IS an order-preserving index into a one-word
// bitmap -- no sort per reference, no rank -> token table (lev_completion.cu)
__device__ __forceinline__ bool lev_tokens_direct(const int* state, int* tmin) {
    const unsigned umax = (unsigned)state[1], umin = ~(unsigned)state[2];
    *tmin = (int)(umin ^ 0x80000000u);
    return !(state[0] & B200LEV_FLAG_WIDE_TOKENS) && umax >= umin && umax - umin < 32u;
}
// the packed mask kernel (lev_mask16.cu) and lev_warp_kernel split a mask-mode batch by these
// two rules: the first is per call, the second per pair
__device__ __forceinline__ bool lev_mask16_tokens_ok(const int* state) {
    return !(state[0] & B200LEV_FLAG_WIDE_TOKENS) && lev_tokens_narrow(state);
}
__device__ __forceinline__ bool lev_mask16_takes(const LevParams& p, int pair) {
    return p.ndist[pair / p.ref_group] <= 32;
}
#endif

// optional per-kernel timing (b200lev_profile): CUDA events recorded on the launch stream
// around each phase; slots of b200lev_profile_read()
enum LevProfSlot { LEV_PROF_PACK_REF = 0, LEV_PROF_PACK_HYP, LEV_PROF_SORT, LEV_PROF_DP,
                   LEV_PROF_FINALIZE, LEV_PROF_STANDBY, LEV_PROF_BV_PROBE, LEV_PROF_BV_DP,
                   LEV_PROF_COMP_UID, LEV_PROF_COMP_FILL, LEV_PROF_ERR_SUM, LEV_PROF_MASK16,
                   LEV_PROF_NSLOTS };
void lev_prof_begin(int slot, cudaStream_t st);
void lev_prof_end(int slot, cudaStream_t st);

// host-side status plumbing (lev_abi.cu)
void lev_set_error(const char* fmt, ...);
int lev_check_cuda(const char* what);

// kernels' host launchers
int lev_launch_pack(const b200lev_tokens_t* t, int has_eos, int64_t eos, int include_eos,
                    int32_t* packed, int64_t Tp, uint16_t* packed16, int64_t Tp16, int32_t* lens,
                    int32_t* flags, int32_t* state, int missing_flag, const int32_t* ref_len,
                    int ref_group, int G, int* ghist, int bv_check, cudaStream_t st,
                    int32_t* split_scratch = nullptr);  // [N + ceil(N / 32)] words, or NULL
int lev_launch_dp(const LevParams& p, int mode, bool count_mode, bool float_path,
                  cudaStream_t st);
int lev_launch_group(const LevParams& p, int mode, bool count_mode, cudaStream_t st);
int lev_launch_mask16(const LevParams& p, bool float_path, cudaStream_t st);
int lev_launch_cta(const LevParams& p, int mode, bool count_mode, bool float_path, cudaStream_t st);
// b200lev_error_counts (p.counts) and b200lev_error_alignment (p.ops and p.trace set): K1 with the
// insertion channel after K0, and for the alignment its choice trace and the walk (lev_dp.cu /
// lev_align.cuh); and the short form for R <= 64, one launch straight from the raw tokens
// (lev_counts.cuh; `p` supplies the costs, the flags and the output)
int lev_launch_counts_dp(const LevParams& p, bool float_path, cudaStream_t st);
int lev_counts_short_launch(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                            const b200lev_opts_t* o, const LevParams& p, bool float_path,
                            cudaStream_t st);
// b200lev_infix (p.out the distances; p.infix_start / p.infix_end with `spans`): K1 with column 0
// pinned to 0, after K0 (lev_dp.cu)
int lev_launch_infix_dp(const LevParams& p, bool float_path, bool spans, cudaStream_t st);
// lanes per pair if the shapes admit the group kernel (its histogram is then built at
// pack time), else 0
int lev_group_eligible(int64_t R, int64_t H, int64_t P);
// Device-side choice between the bit-vector path and the wavefront path (no host round trip).
// When the shapes and costs admit the n-best bit-vector kernel it is enqueued FIRST: its probe
// looks at a sample of the blocks of 32 consecutive pairs for more than 4 runs of identical
// references (n-best batches have at most 4) and vetoes through state[3] if it finds one; every
// kernel of the wavefront path, enqueued behind, then starts with lev_bv_took() and exits at
// once if the work is already done (and the bit-vector kernel with the opposite test).
__device__ __forceinline__ bool lev_bv_took(const int* state) {
    return *reinterpret_cast<const volatile int*>(state + 3) == 0;
}
// unit-cost bit-vector path (lev_bitvec.cu): which kernel takes a final / prefix call
enum LevBvRoute {
    LEV_BV_NONE,      // the wavefront path alone
    LEV_BV_SHORT,     // Ks takes the call (and, in final mode, the error sums)
    LEV_BV_FUSED,     // Kb takes the call
    LEV_BV_SELECTED,  // probe + Kb ahead of the wavefront path's stand-by chain (lev_bv_took)
};
// `p` as lev_abi.cu fills it for the call: costs, shapes, ref_group, out_sn
LevBvRoute lev_bitvec_route(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp, int mode,
                            const LevParams& p, bool count_mode, bool float_path);
// `ws` is the aligned workspace laid out as `L`; `acc` (final mode, may be NULL) goes to Ks.
// With LEV_BV_SELECTED `after_probe` (a cudaEvent_t, may be NULL) is recorded once the veto is final.
// cross_b > 0 (LEV_BV_SHORT, final mode; b200lev_final_cross): `hyp` is the expanded (H, G*A*B) view
// of the (H, G*B) hypotheses and Ks reads hypothesis column (p / (A*B)) * B + p % B for pair p.
int lev_bitvec_launch(LevBvRoute route, const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                      const b200lev_opts_t* o, int mode, const LevLayout& L, char* ws,
                      const LevParams& p, cudaStream_t st, void* after_probe, double* acc,
                      int64_t cross_a = 0, int64_t cross_b = 0);
// b200lev_final_cross, gather path: out (H, G*A*B), sequence-first and contiguous, column p =
// hypothesis column (p / (A*B)) * B + p % B of `hyp` (any strides), same element width
int lev_launch_cross_gather(const b200lev_tokens_t* hyp, int64_t A, int64_t B, int64_t P, void* out,
                            cudaStream_t st);
// K7 (lev_loss.cu): acc[0] += sum(er), acc[1] += sum of the pairs' reference lengths, acc[2] += P
// (P >= 1, ref_group >= 1)
int lev_launch_err_sum(const float* er, const int32_t* ref_lens, int64_t P, int ref_group,
                       double* acc, cudaStream_t st);
int lev_launch_uid(const b200lev_tokens_t* ref, const int32_t* packed, const int* state,
                   const int32_t* ref_len, int32_t* uid,
                   int64_t* dtok, int32_t* ndist, int64_t Rp, cudaStream_t st);
int lev_launch_completion_fill(const uint32_t* dbits, const int64_t* dtok, const int* state, int64_t Rp,
                               int64_t Hout, int64_t P, int64_t Wd, int ref_group, int64_t U,
                               int64_t padding, int64_t* out, int64_t out_si, int64_t out_sn,
                               cudaStream_t st);
