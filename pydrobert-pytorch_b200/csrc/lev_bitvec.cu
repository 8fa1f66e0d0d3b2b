// lev_bitvec.cu -- unit-cost fast path: which bit-parallel kernel, if any, takes a call.
//
// When ins == del == sub (SM:168-174 reduces that case to unit costs and a multiplier) the
// DP row of SM:286-350 is determined by its +1/0/-1 differences, and Myers' bit-vector
// recurrence (J. ACM 46(3), 1999; Hyyro's edit-distance form) advances a whole row of up to
// 32*W reference positions with ~10 logic operations per 32-bit word instead of ~2.5
// instructions per CELL in the packed wavefront kernel (lev_group.cu).  The value the
// reference reads off each row -- column r, the distance between the full reference and a
// hypothesis prefix (SM:352-358, 386-405) -- is the running score of the recurrence, so
// the final and the prefix modes both fall out of one pass over the hypothesis.  Both kernels
// work with lane = pair straight from the raw sequence-first tokens; K0 (lev_pack.cu) is not
// needed on this path.
//
// Eligibility (lev_bitvec_route): unit costs after SM:168-174, final or prefix mode, at most
// 128 reference positions, unit stride along the batch axis of both token tensors and of the
// prefix output.  Then, per call:
//
//   Ks  lev_bv_short_kernel (lev_bvshort.cu), R <= 64: the reference in registers, no tables --
//       any batch, taken unconditionally.
//   Kb  lev_bv_fused_kernel (lev_bvfused.cu), R <= 128: per-run hash tables and match masks in
//       shared memory, built for n-best batches (<= 4 distinct references per 32 pairs).  A call
//       that declares its references shared (ref_group >= 8) takes it unconditionally; any other
//       batch of at least B200LEV_BITVEC_MIN_PAIRS pairs whose wavefront path is the group kernel
//       is enqueued AHEAD of that path and decided on the device: lev_bv_probe_kernel vetoes
//       through state[3] (lev_bv_took, lev_common.cuh) when a sampled block holds more references
//       than that, and the wavefront kernels -- which otherwise exit at once -- do the work.
#include "lev_bitvec.cuh"

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// B200LEV_BITVEC: 0 = never, 1 = forced (tests: whatever the references look like, multi-pass
// where a block of 32 pairs holds more than 4 distinct references), default 2 = enqueued ahead
// of the wavefront path, which it pre-empts on the device when the batch is n-best shaped.
static int lev_bitvec_mode() {
    const char* e = getenv("B200LEV_BITVEC");
    return e != nullptr ? atoi(e) : 2;
}
static int64_t lev_bv_min_pairs() {
    int64_t v = 1024;  // below this the warp-per-pair kernels have the lower latency
    if (const char* e = getenv("B200LEV_BITVEC_MIN_PAIRS")) v = atoll(e);
    return v;
}

// the short-reference form (lev_bvshort.cu) is ONE launch with nothing to set up: it serves every
// batch size (32 pairs of 50 tokens: 34 us for the whole call against 41 us through pack + DP)
static int64_t lev_bvshort_min_pairs() {
    int64_t v = 1;
    if (const char* e = getenv("B200LEV_BVSHORT_MIN_PAIRS")) v = atoll(e);
    return v;
}

// `grouped`: the call says how its references are shared (ref_group hypotheses per reference,
// _string.py:1426/1439 -- minimum_error_rate_loss): with 8 or more a block of 32 pairs holds at
// most 4 - 5 references, which is what the fused kernel's tables are built for, so there is
// nothing to probe and no stand-by chain to enqueue; such a call is worth it from a few warps on.
LevBvRoute lev_bitvec_route(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp, int mode,
                            const LevParams& p, bool count_mode, bool float_path) {
    const int bv = lev_bitvec_mode();
    if (bv == 0 || mode == LEV_MODE_MASK) return LEV_BV_NONE;
    if (count_mode || float_path || p.ins_i != 1 || p.del_i != 1 || p.sub_i != 1) return LEV_BV_NONE;
    // (lev_layout has a block counter for R <= 128 only)
    if (ref->T > 128 || ref->T < 1 || hyp->T >= (1 << 20)) return LEV_BV_NONE;
    if (!lev_bvfused_supports(ref->elem_bytes) || ref->elem_bytes != hyp->elem_bytes) return LEV_BV_NONE;
    const bool short_form = lev_bvshort_supports(ref->elem_bytes, ref->T) && hyp->N >= lev_bvshort_min_pairs();
    const bool grouped = !short_form && p.ref_group >= 8 && hyp->N >= 128;
    if (!short_form && !grouped && hyp->N < lev_bv_min_pairs()) return LEV_BV_NONE;
    if (ref->stride_t >= ((int64_t)1 << 31) || hyp->stride_t >= ((int64_t)1 << 31) ||
        ref->stride_t < 0 || hyp->stride_t < 0)
        return LEV_BV_NONE;
    if ((ref->N > 1 && ref->stride_n != 1) || (hyp->N > 1 && hyp->stride_n != 1)) return LEV_BV_NONE;
    if (mode == LEV_MODE_PREFIX && p.out_sn != 1) return LEV_BV_NONE;
    // the short-reference kernel takes any batch, the fused kernel any batch whose references the
    // caller declared shared: nothing to select on the device, no chain behind them
    if (short_form) return LEV_BV_SHORT;
    if (grouped || bv == 1) return LEV_BV_FUSED;
    // device-selected: only where the wavefront fallback is the group path, whose kernels know how
    // to stand by
    return lev_group_eligible(p.R, p.H, p.P) ? LEV_BV_SELECTED : LEV_BV_NONE;
}

int lev_bitvec_launch(LevBvRoute route, const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                      const b200lev_opts_t* o, int mode, const LevLayout& L, char* ws,
                      const LevParams& p, cudaStream_t st, void* after_probe, double* acc,
                      int64_t cross_a, int64_t cross_b) {
    LevBvArgs a;
    memset(&a, 0, sizeof(a));
    a.ref = ref->data;
    a.hyp = hyp->data;
    a.ref_st = ref->stride_t;
    a.hyp_st = hyp->stride_t;
    a.R = (int)ref->T;
    a.H = (int)hyp->T;
    a.P = (int)hyp->N;
    a.ref_group = o->ref_group;
    a.has_eos = o->has_eos;
    a.eos = o->eos;
    a.include_eos = o->include_eos;
    a.ref_len = (int32_t*)(ws + L.off_ref_len);
    a.hyp_len = (int32_t*)(ws + L.off_hyp_len);
    a.counter = (int*)(ws + L.off_bv_counter);
    a.flags = p.flags;
    // buckets of 4 ways: on average at most one token per bucket; a key's low s bits hold a
    // position or R (no match), so 2^s > R
    a.slots_log2 = 4;
    while ((1 << a.slots_log2) <= a.R) ++a.slots_log2;
    a.mode = mode;
    a.norm = o->norm;
    a.exclude_last = mode == LEV_MODE_PREFIX ? o->exclude_last : 0;
    a.Hout = p.Hout;
    a.mult = p.mult;
    a.padding = (float)o->padding;
    a.out = p.out;
    a.out_si = p.out_si;
    if (route == LEV_BV_SHORT) {  // R <= 64: lane = pair, reference in registers, no tables (lev_bvshort.cu)
        a.acc = mode == LEV_MODE_FINAL ? acc : nullptr;
        a.cross_ab = (int)(cross_a * cross_b);  // (< 2^31: b200lev_final_cross bounds the pairs)
        a.cross_b = (int)cross_b;
        if (getenv("B200LEV_TRACE"))
            fprintf(stderr, "b200lev: short bit-vector kernel, mode %d, R=%d H=%d P=%d\n", mode, a.R, a.H, a.P);
        return lev_bvshort_launch(a, ref->elem_bytes, st);
    }
    if (route == LEV_BV_SELECTED) {
        // Kb runs only if its probe does not veto.  The state words are cleared here, once, for
        // both paths: the wavefront chain's pack kernels find them cleared.
        a.state = (int32_t*)(ws + L.off_flags);
        a.check_state = 1;
        if (cudaMemsetAsync(a.state, 0, sizeof(int32_t) * (size_t)(4 + L.nbins), st) != cudaSuccess)
            return lev_check_cuda("memset");
    }
    if (getenv("B200LEV_TRACE"))
        fprintf(stderr, "b200lev: fused bit-vector kernel, mode %d, R=%d H=%d P=%d W=%d device-selected=%d\n",
                mode, a.R, a.H, a.P, (a.R + 31) / 32, a.check_state);
    return lev_bvfused_launch(a, ref->elem_bytes, st, after_probe);
}
