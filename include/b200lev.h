/*
 * b200lev.h -- C ABI of the B200-native Levenshtein hot path (libb200lev.so).
 *
 * Drop-in boundary for the string-matching path of sdrobert/pydrobert-pytorch
 * ("SM" = src/pydrobert/torch/_string.py of the reference).  The reference has no
 * FFI of its own -- its boundary is the Python call surface -- so each entry point
 * names the reference function whose body it replaces.  The binding a maintainer
 * would add to the reference (a ctypes stub inside `_string.py`) is shown in
 * INTEGRATION.md; pydrobert-pytorch_b200/b200lev/_abi.py is that binding, complete.
 *
 * Conventions
 *  - plain C types, raw DEVICE pointers, element strides, a cudaStream_t passed as
 *    void*; no torch types.  Nothing here allocates device memory: the caller
 *    supplies outputs and a scratch workspace sized by *_workspace_bytes().
 *  - every call only enqueues work on `stream` (asynchronous w.r.t. the host) and
 *    returns B200LEV_OK, or a negative status with a message retrievable through
 *    b200lev_last_error() (thread-local).  There is NO CPU fallback: without a CUDA
 *    device every compute entry point fails with B200LEV_ERR_CUDA.
 *  - token tensors are borrowed, never written; integer element types of 1, 2, 4 or
 *    8 bytes (signed) are accepted, int64 being the reference's ("long tensor",
 *    SM:588-596).
 *  - `flags` (device int32[1], may be NULL) receives an OR of B200LEV_FLAG_*: the
 *    data-dependent conditions behind the reference's three warnings (the host
 *    reads it back only when `warn=True`, one 4-byte D2H) and behind the error the
 *    reference raises for a loss target that is not a class.
 */
#ifndef B200LEV_H_
#define B200LEV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200LEV_ABI_VERSION 3

#define B200LEV_OK 0
#define B200LEV_ERR_ARG (-1)       /* bad argument (shape, stride, dtype, NULL) */
#define B200LEV_ERR_CUDA (-2)      /* CUDA runtime error / no device */
#define B200LEV_ERR_WORKSPACE (-3) /* workspace too small */
#define B200LEV_ERR_UNSUPPORTED (-4)

/* SM:202-217 (include_eos but no eos in a ref / hyp transcript), SM:361-366 and
 * SM:398-404 (empty reference with norm), and "a token does not fit in int32" (the
 * kernels then take the 64-bit compare path). */
#define B200LEV_FLAG_REF_NO_EOS 1
#define B200LEV_FLAG_HYP_NO_EOS 2
#define B200LEV_FLAG_EMPTY_REF 4
#define B200LEV_FLAG_WIDE_TOKENS 8
/* b200lev_ocd_forward: a target outside [0, V) other than ignore_index (torch's cross_entropy
 * raises "Target t is out of bounds."); the kernels skip such targets and read nothing for them */
#define B200LEV_FLAG_BAD_TARGET 16

/* A borrowed, strided 2-D token view: element (t, n) of a (T, N) "sequence first"
 * tensor lives at data + (t*stride_t + n*stride_n) * elem_bytes.  A batch_first
 * tensor is passed with the two strides swapped (the transpose at SM:181-183). */
typedef struct b200lev_tokens {
    const void *data;
    int32_t elem_bytes; /* 1, 2, 4 or 8 (signed integers) */
    int64_t T;          /* padded sequence length */
    int64_t N;          /* number of sequences */
    int64_t stride_t;
    int64_t stride_n;
} b200lev_tokens_t;

/* The knobs of SM:146-163 (_string_matching). */
typedef struct b200lev_opts {
    int32_t has_eos;     /* eos is not None */
    int64_t eos;
    int32_t include_eos;
    float ins_cost, del_cost, sub_cost;
    int32_t norm;
    int32_t exclude_last;
    int64_t padding;         /* prefix tail fill / completion fill value */
    int32_t return_mistakes; /* 1 for the *error_rate* family, 0 for *edit_distance* */
    int32_t ref_group;       /* >= 1: pair n reads reference column n / ref_group (the
                                n-best repeat of SM:1426,1439 without materialising it) */
} b200lev_opts_t;

int b200lev_abi_version(void);
const char *b200lev_last_error(void);
/* number of CUDA devices visible to the library (0 => every compute call fails) */
int b200lev_device_count(void);

/* Scratch bytes needed by the calls below for these shapes (packed tokens, lengths,
 * bucketing tables).  kind: B200LEV_WS_FINAL for b200lev_final*, B200LEV_WS_PREFIX for
 * b200lev_prefix (adds the raw prefix rows), B200LEV_WS_COMPLETION for the completion
 * calls (adds the distinct-token tables and bitmaps), B200LEV_WS_ALIGN for
 * b200lev_error_alignment (adds every DP cell's 2-bit choice).  The alignment kind adds, for
 * ref->T <= 64 with equal token widths, 8 or 16 bytes per hypothesis position and pair (R <= 32
 * or not); otherwise (H + 31) * 64 * ceil((R + 1) / 256) bytes or (H + 31) * 32 *
 * ceil((R + 1) / 128) bytes per pair, whichever is larger, plus one int32 per pair: about
 * 15 kB per pair at R = H = 200, 1 MB at R = H = 2000. */
#define B200LEV_WS_FINAL 0
#define B200LEV_WS_COMPLETION 1
#define B200LEV_WS_PREFIX 2
#define B200LEV_WS_ALIGN 3
size_t b200lev_workspace_bytes(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                               int32_t kind, int32_t exclude_last);

/*
 * error_rate (SM:409-434) / edit_distance (SM:437-461): one fp32 value per pair.
 *   out: device float[hyp->N]
 */
int b200lev_final(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                  const b200lev_opts_t *opts, float *out, void *workspace,
                  size_t workspace_bytes, int32_t *flags, void *stream);

/*
 * Every reference of a group against every hypothesis of it: ref holds G groups of A sequences
 * (ref->N = G*A, reference (g, a) is column g*A + a) and hyp G groups of B (hyp->N = G*B,
 * hypothesis (g, b) is column g*B + b).  out[(g*A + a)*B + b] is b200lev_final of reference
 * column g*A + a against hypothesis column g*B + b with the same opts, bit for bit, without the
 * cross product being materialised by the caller.  opts as for b200lev_final; ref_group must be 1.
 * G*A*B must be below 2^31.  Where b200lev_final would send the expanded pairs to the short-reference
 * kernel (unit costs after SM:168-174, ref->T <= 64, equal token widths, unit batch strides) that
 * kernel reads the hypotheses in place; otherwise the expanded (hyp->T, G*A*B) hypotheses are
 * gathered into the workspace first.  out: device float[G*A*B].
 * Workspace: b200lev_final_cross_workspace_bytes(ref, hyp, A, B, opts) -- the costs decide the
 * route and so the size; it is b200lev_workspace_bytes of the expanded pairs, plus
 * hyp->T * G*A*B * hyp->elem_bytes (rounded up) and 128 bytes on the gather route.
 */
size_t b200lev_final_cross_workspace_bytes(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                                           int64_t A, int64_t B, const b200lev_opts_t *opts);
int b200lev_final_cross(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp, int64_t A, int64_t B,
                        const b200lev_opts_t *opts, float *out, void *workspace, size_t workspace_bytes,
                        int32_t *flags, void *stream);

/*
 * prefix_error_rates (SM:520-550) / prefix_edit_distances (SM:553-583).
 *   out: device float, element (i, n) at out[i*out_stride_i + n*out_stride_n],
 *        i in [0, H+1) or [0, H) when exclude_last.
 */
int b200lev_prefix(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                   const b200lev_opts_t *opts, float *out, int64_t out_stride_i,
                   int64_t out_stride_n, void *workspace, size_t workspace_bytes,
                   int32_t *flags, void *stream);

/*
 * Per pair the correct / substitution / deletion / insertion counts (sclite's C/S/D/I) along
 * the path the count mode of error_rate takes (SM:292-314: sub over ins over del on ties), also
 * for uniform costs.  S + D + I equals error_rate(norm=False) for the same eos and costs,
 * C + S + D the reference length and C + S + I the hypothesis length.
 * out: device int64, element (n, k) at out[n*4 + k], k = 0 correct, 1 substitutions,
 * 2 deletions, 3 insertions.  opts: has_eos, eos, include_eos and the costs as for
 * b200lev_final; ref_group must be 1; norm, exclude_last, padding, return_mistakes are
 * ignored.  Workspace: b200lev_workspace_bytes(ref, hyp, B200LEV_WS_FINAL, 0).
 */
int b200lev_error_counts(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                         const b200lev_opts_t *opts, int64_t *out, void *workspace,
                         size_t workspace_bytes, int32_t *flags, void *stream);

/*
 * The edit operations along the path b200lev_error_counts counts, one per step, in forward
 * order from the start of both sequences to cell (h, r): 0 correct, 1 substitution,
 * 2 deletion, 3 insertion.  Row 0 of the DP is all deletions and column 0 all insertions.
 * Per pair the histogram of the ops equals b200lev_error_counts with the same arguments.
 * out: device int8, step k of pair n at out[k*out_stride_k + n*out_stride_n], k in
 * [0, ref->T + hyp->T); steps from the path length r + I on hold -1.  opts as for
 * b200lev_error_counts (ref_group must be 1).
 * Workspace: b200lev_workspace_bytes(ref, hyp, B200LEV_WS_ALIGN, 0).
 */
int b200lev_error_alignment(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                            const b200lev_opts_t *opts, int8_t *out, int64_t out_stride_k,
                            int64_t out_stride_n, void *workspace, size_t workspace_bytes,
                            int32_t *flags, void *stream);

/*
 * Infix edit distance: per pair the cheapest alignment of the whole reference against any
 * contiguous stretch hyp[s:e] of the hypothesis, leading and trailing hypothesis tokens free.
 * D is the DP of b200lev_final (same lengths, costs, uniform-cost shortcut and fp32 operation
 * order) with one change: column 0 is 0 on every row (row 0 keeps D[0][j] = j deletions).
 *   dist : device float[hyp->N], the minimum over 0 <= i <= h of D[i][r]; opts->norm divides it
 *          by r as b200lev_final does (an empty reference has distance 0, and raises
 *          B200LEV_FLAG_EMPTY_REF under norm).
 *   start, end : device int64[hyp->N], both NULL (distances only) or both set.  end is the
 *          smallest row reaching the minimum, start the start row of the optimal path into
 *          (end, r): leaving column 0 at row s starts at s, and at each cell the largest start
 *          among the predecessors (diagonal, up, deletion run origin) reaching its value wins.
 *          The match is hyp[start:end].  Not with opts->norm.
 * opts: has_eos, eos, include_eos, the costs and norm as for b200lev_final; ref_group must be 1;
 * exclude_last, padding and return_mistakes are ignored.  Free ends on the reference side
 * instead: swap ref and hyp, and ins_cost and del_cost.
 * Workspace: b200lev_workspace_bytes(ref, hyp, B200LEV_WS_FINAL, 0).
 */
int b200lev_infix(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                  const b200lev_opts_t *opts, float *dist, int64_t *start, int64_t *end,
                  void *workspace, size_t workspace_bytes, int32_t *flags, void *stream);

/*
 * optimal_completion (SM:464-517), two phases around the one host read the
 * reference also needs (SM:511: U = counts.max().item()).
 *   phase 1 runs the DP in mask mode (SM:271-278, 319-339, 347-355), leaves the
 *           per-prefix sets in the workspace and writes U to *umax (device int32[1]);
 *   phase 2 expands them into out (int64, element (i, n, u) at
 *           out[i*stride_i + n*stride_n + u]), ascending, padded with opts->padding.
 * The same workspace must be passed to both phases.
 */
int b200lev_completion_count(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                             const b200lev_opts_t *opts, void *workspace,
                             size_t workspace_bytes, int32_t *umax, int32_t *flags,
                             void *stream);
int b200lev_completion_fill(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                            const b200lev_opts_t *opts, const void *workspace,
                            size_t workspace_bytes, int64_t U, int64_t *out,
                            int64_t out_stride_i, int64_t out_stride_n, void *stream);

/* floating-point element types of the loss entry points */
#define B200LEV_F32 0
#define B200LEV_F16 1
#define B200LEV_BF16 2
#define B200LEV_F64 3

#define B200LEV_REDUCE_NONE 0
#define B200LEV_REDUCE_MEAN 1
#define B200LEV_REDUCE_SUM 2

/*
 * hard_optimal_completion_distillation_loss (SM:1229-1251) given the targets of
 * optimal_completion(padding=ignore_index, exclude_last=True).
 *   logits : (A, B, V) element (a, b, v) at logits[a*ls_a + b*ls_b + v]   (dtype code)
 *   targets: int64 (A, B, U) element at targets[a*ts_a + b*ts_b + u]
 *   weight : NULL or V class weights in the ACCUMULATION type (see below): float[V], or
 *            double[V] when dtype is F64
 *   seq_axis: 0 if A is the hypothesis axis (seq-first), 1 if B is (batch_first)
 * Scratch/outputs are in the ACCUMULATION type: fp32, or fp64 when dtype is F64.
 * Forward writes per[A*B] (row-major (a, b)), lse[A*B], and -- for mean/sum -- the
 * scalar loss[0] plus denom[] (per-sequence number of steps with targets, length =
 * size of the non-sequence axis).  Backward reads grad_out (accumulation type; one
 * element for mean/sum, A*B for none) and writes grad_logits (dtype of logits,
 * contiguous (A, B, V)).  A target outside [0, V) other than ignore_index is skipped; the
 * forward ORs B200LEV_FLAG_BAD_TARGET into *flags (device int32[1], may be NULL) for it.
 */
int b200lev_ocd_forward(const void *logits, int32_t dtype, int64_t A, int64_t B, int64_t V,
                        int64_t ls_a, int64_t ls_b, const int64_t *targets, int64_t U,
                        int64_t ts_a, int64_t ts_b, const void *weight,
                        int64_t ignore_index, int32_t reduction, int32_t seq_axis,
                        void *per, void *lse, void *denom, void *loss, int32_t *flags,
                        void *stream);
int b200lev_ocd_backward(const void *logits, int32_t dtype, int64_t A, int64_t B, int64_t V,
                         int64_t ls_a, int64_t ls_b, const int64_t *targets, int64_t U,
                         int64_t ts_a, int64_t ts_b, const void *weight,
                         int64_t ignore_index, int32_t reduction, int32_t seq_axis,
                         const void *lse, const void *denom, const void *grad_out,
                         void *grad_logits, void *stream);

/*
 * minimum_error_rate_loss epilogue (SM:1463-1471) on the (N, M) error rates.
 *   er: float[N*M] from b200lev_final; log_probs (N, M) strided, dtype code.
 * Forward writes per[N*M] and, for mean/sum, loss[0] (accumulation type, see above).
 * Backward writes grad[N*M] (dtype of log_probs, contiguous).
 */
int b200lev_mwer_forward(const float *er, const void *log_probs, int32_t dtype, int64_t N,
                         int64_t M, int64_t lp_sn, int64_t lp_sm, int32_t sub_avg,
                         int32_t reduction, void *per, void *loss, void *stream);
int b200lev_mwer_backward(const float *er, const void *log_probs, int32_t dtype, int64_t N,
                          int64_t M, int64_t lp_sn, int64_t lp_sm, int32_t sub_avg,
                          int32_t reduction, const void *grad_out, void *grad, void *stream);

/*
 * Minimum-Bayes-risk selection over N n-best lists of M hypotheses (decoding only, no gradient).
 *   er: float[N*M*M] from b200lev_final_cross of the hypotheses against themselves (A = B = M):
 *       er[(n*M + a)*M + i] scores hypothesis i against hypothesis a as the reference.
 *   log_probs (N, M) strided, dtype code.
 * p = softmax(log_probs[n]) in the accumulation type (fp32; fp64 for F64), rounded to the dtype;
 * risk[n*M + i] = sum over a of p_a * er[n, a, i] (dtype of log_probs, contiguous (N, M)); every
 * column is summed in the same order, so identical hypotheses get bitwise identical risks.
 * best[n] (int64) = the arg min of risk[n, :], equal risks to the lowest index.  M >= 1.
 */
int b200lev_mbr(const float *er, const void *log_probs, int32_t dtype, int64_t N, int64_t M,
                int64_t lp_sn, int64_t lp_sm, void *risk, int64_t *best, void *stream);

/* b200lev_final and the bulk-scoring totals in one call: `out` as b200lev_final, and
 * acc[0] += sum(out), acc[1] += sum over pairs of the reference length, acc[2] += #pairs (fp64
 * on the device, so one all-reduce(sum) of 24 bytes finishes a multi-GPU job).  Where the
 * short-reference kernel serves the call the sums are accumulated inside it (no second kernel):
 * the per-batch body of command_line.py:1124-1147. */
int b200lev_final_sums(const b200lev_tokens_t *ref, const b200lev_tokens_t *hyp,
                       const b200lev_opts_t *opts, float *out, void *workspace,
                       size_t workspace_bytes, int32_t *flags, double *acc, void *stream);

/* fill_after_eos (SM:30-42), the scan: tokens is a contiguous int64 (outer, T, inner)
 * view; mask[o, t, i] = 1 iff an eos occurs at some t' < t.  The broadcasted fill of
 * SM:42 is a masked_fill with this mask on the caller's side. */
int b200lev_after_eos_mask(const int64_t *tokens, int64_t outer, int64_t T, int64_t inner,
                           int64_t eos, unsigned char *mask, void *stream);

/* Bulk-scoring batches ("next #2" of the hot-path scope): what command_line.py:1110-1121 builds
 * on the host with torch.tensor(transcript + [eos]) per utterance and pad_sequence.  The
 * corpus is flat (tokens of elem_bytes 2, 4 or 8; offsets[k] .. offsets[k+1] = utterance k);
 * row u of out (n, T) row-major = utterance sel[u] (u if sel is NULL), then eos, then pad.
 * T must exceed every selected utterance's length.  All pointers are device pointers. */
int b200lev_ragged_to_padded(const void *flat, int32_t elem_bytes, const int64_t *offsets,
                             const int64_t *sel, int64_t n, int64_t T, int64_t eos, int64_t pad,
                             void *out, void *stream);

/* sequence_log_probs, tensor path (_decoding.py:1516-1548; "next #1" of the hot-path scope):
 *   out[a, b] = sum over the steps t that count of log_softmax(logits[a, t, b, :])[hyp[a, t, b]]
 * A step counts if its token lies in [0, V) and t <= the first eos of the sequence (a, b)
 * (has_eos; the eos step itself counts).  logits: contiguous (outer, T, inner, V) of `dtype`
 * (B200LEV_F32/F16/BF16/F64); hyp: contiguous int64 (outer, T, inner); out: (outer, inner) in
 * the dtype of logits.  Scratch supplied by the caller: len int32[outer*inner]; row_lp and
 * row_lse, (outer*T*inner) elements of the ACCUMULATION type (fp32; fp64 for F64) -- row_lse and
 * len are what the backward call needs.  Backward: grad_logits (same shape/dtype as logits) =
 * grad_out[a, b] * (onehot(hyp) - softmax) on the steps that count, 0 elsewhere. */
int b200lev_seqlp_forward(const void *logits, int32_t dtype, int64_t outer, int64_t T,
                          int64_t inner, int64_t V, const int64_t *hyp, int32_t has_eos,
                          int64_t eos, int32_t *len, void *row_lp, void *row_lse, void *out,
                          void *stream);
int b200lev_seqlp_backward(const void *logits, int32_t dtype, int64_t outer, int64_t T,
                           int64_t inner, int64_t V, const int64_t *hyp, const int32_t *len,
                           const void *row_lse, const void *grad_out, void *grad_logits,
                           void *stream);

/* ctc_greedy_search (_decoding.py:507-560; "next #4" of the hot-path scope).  logits:
 * contiguous (outer, T, inner, V) of `dtype`; sequence q = (a, b) of (outer, inner); in_lens:
 * int64[outer*inner] or NULL (every step valid); blank in [0, V).  Outputs: paths int64
 * (outer, T, inner) = the arg max per step with blanks and repeats dropped, compacted to the
 * front (positions >= out_lens keep the raw arg max, as the reference's masked_scatter_
 * does); out_lens int64[outer*inner]; max_out[outer*inner] in the dtype of logits = the sum
 * over valid steps of max(log_softmax) -- or, with is_probs, the product of the maxima.
 * Scratch: arg int64 and row_val, row_lse accumulation-type (fp32; fp64 for F64), all
 * (outer*T*inner); len int32[outer*inner] (clamped in_lens).  arg, row_lse and len are what
 * b200lev_seqlp_backward needs (hyp := arg) for the gradient of max_out w.r.t. the logits. */
int b200lev_ctc_greedy(const void *logits, int32_t dtype, int64_t outer, int64_t T, int64_t inner,
                       int64_t V, const int64_t *in_lens, int64_t blank, int32_t is_probs,
                       int64_t *arg, void *row_val, void *row_lse, int32_t *len, int64_t *paths,
                       int64_t *out_lens, void *max_out, void *stream);

/* Host-side plumbing for callers whose tensors live in HOST memory (the reference API accepts
 * CPU tensors: SM:146 has no device requirement): one strided 2-D copy between host and
 * device on `stream`, so that a caller can move a COLUMN block of a (T, N) tensor -- all
 * positions of a slice of the batch -- with one DMA and overlap the copies of block k+1,
 * the kernels of block k and the read-back of block k-1 on three streams.  Pitches and
 * width in bytes; to_device != 0: host -> device, else device -> host.  The copy is
 * asynchronous when the host side is page-locked. */
int b200lev_copy2d_async(void *dst, size_t dst_pitch, const void *src, size_t src_pitch,
                         size_t width_bytes, size_t height, int32_t to_device, void *stream);

/* Optional per-kernel timing for bench.py: when enabled, every phase of the calls above is
 * bracketed by CUDA events on the launch stream.  b200lev_profile_read waits for the last
 * recorded events and returns milliseconds (or -1) for the slots
 *   0 pack(ref)  1 pack(hyp)  2 bucketing (sort)  3 DP kernel(s)  4 prefix finalize
 *   5 stand-by 64-bit-token kernel. */
int b200lev_profile(int enable);
int b200lev_profile_read(float *ms, int n);

/* INT32 issue-rate microbenchmark used for the roofline denominator (bench.py):
 * runs `iters` dependent-free VIADDMNMX/IADD3 per thread on `blocks` x 256 threads and
 * returns the op count through *ops (host).  Timed by the caller with CUDA events. */
int b200lev_int32_peak_kernel(int32_t variant, int64_t blocks, int64_t iters, int32_t *sink,
                              double *ops, void *stream);

/* ---- N-best producers' step functions (SURVEY 8f #3) -------------------------------------
 * b200lev_beam_topk   -- the top-k of reference _decoding.py:117-121 (beam_search_advance):
 *   candidates log_probs_prev[n, k] + log_probs_t[n, k, v] (summed and rounded in the tensors'
 *   dtype: 0 fp32, 1 fp16, 2 bf16, 3 fp64; element strides), the `width` best per batch element
 *   in descending order, equal scores by ascending flat index k * V + v.  Writes
 *   log_probs_next (N, width) in the same dtype, next_src (N, width) = k and y_t (N, width) = v
 *   (int64); columns beyond min(width, Kp * V) get -inf / 0 / 0 (_decoding.py:143-152).
 * b200lev_path_extend -- the gather / cat / scatter of _decoding.py:123-141 (and of
 *   random_walk_advance, _decoding.py:1268-1281, with src = NULL): y_next (S_out, N, W) from
 *   y_prev (S, N, Kp), both contiguous int64; src (N, W) or NULL (identity), lens_prev (N, Kp)
 *   or NULL (all S), y_t (N, W); S_out is S or S + 1; lens_next (N, W) may be NULL.  Columns
 *   k >= K are padding (zeros; the reference leaves them uninitialised).
 */
int b200lev_beam_topk(const void *log_probs_t, int32_t dtype, int64_t N, int64_t Kp, int64_t V,
                      int64_t stride_n, int64_t stride_k, int64_t stride_v,
                      const void *log_probs_prev, int64_t prev_stride_n, int64_t prev_stride_k,
                      int64_t width, void *log_probs_next, int64_t *next_src, int64_t *y_t,
                      void *stream);
int b200lev_path_extend(const int64_t *y_prev, int64_t S, int64_t N, int64_t Kp, const int64_t *src,
                        const int64_t *lens_prev, const int64_t *y_t, int64_t K, int64_t W,
                        int64_t S_out, int64_t *y_next, int64_t *lens_next, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200LEV_H_ */
