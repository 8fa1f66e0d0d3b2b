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
// Eligibility (lev_bitvec_eligible): unit costs after SM:168-174, final or prefix mode, at most
// 128 reference positions, unit stride along the batch axis of both token tensors and of the
// prefix output.  Then, per call:
//
//   Ks  lev_bv_short_kernel (lev_bvshort.cu), R <= 64: the reference in registers, no tables --
//       any batch, taken unconditionally.
//   Kb  lev_bv_fused_kernel (lev_bvfused.cu), R <= 128: per-run hash tables and match masks in
//       shared memory, built for n-best batches (<= 4 distinct references per 32 pairs).  A call
//       that declares its references shared (ref_group >= 8) takes it unconditionally; any other
//       batch of at least B200LEV_BITVEC_MIN_PAIRS pairs is enqueued AHEAD of the wavefront path
//       and decided on the device: lev_bv_probe_kernel vetoes through state[3] (lev_bv_took,
//       lev_common.cuh) when a sampled block holds more references than that, and the wavefront
//       kernels -- which otherwise exit at once -- do the work.
#include "lev_bitvec.cuh"

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
// B200LEV_BITVEC: 0 = never, 1 = forced (tests: whatever the references look like, multi-pass
// where a block of 32 pairs holds more than 4 distinct references), default 2 = enqueued ahead
// of the wavefront path, which it pre-empts on the device when the batch is n-best shaped.
int lev_bitvec_mode() {
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
bool lev_bitvec_eligible(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp, int mode,
                         bool count_mode, bool float_path, int ins_i, int del_i, int sub_i,
                         int64_t out_sn, int ref_group, bool* short_form, bool* grouped) {
    *short_form = false;
    *grouped = false;
    if (lev_bitvec_mode() == 0) return false;
    if (mode != LEV_MODE_FINAL && mode != LEV_MODE_PREFIX) return false;
    if (count_mode || float_path || ins_i != 1 || del_i != 1 || sub_i != 1) return false;
    if (ref->T > 128 || ref->T < 1 || hyp->T >= (1 << 20)) return false;
    if (!lev_bvfused_supports(ref->elem_bytes) || ref->elem_bytes != hyp->elem_bytes) return false;
    *short_form = lev_bvshort_supports(ref->elem_bytes, ref->T) && hyp->N >= lev_bvshort_min_pairs();
    *grouped = !*short_form && ref_group >= 8 && hyp->N >= 128;
    if (!*short_form && !*grouped && hyp->N < lev_bv_min_pairs()) return false;
    if (ref->stride_t >= ((int64_t)1 << 31) || hyp->stride_t >= ((int64_t)1 << 31) ||
        ref->stride_t < 0 || hyp->stride_t < 0)
        return false;
    if ((ref->N > 1 && ref->stride_n != 1) || (hyp->N > 1 && hyp->stride_n != 1)) return false;
    if (mode == LEV_MODE_PREFIX && out_sn != 1) return false;
    return true;
}

// The caller has checked lev_bitvec_eligible.  `counter` is one workspace word (Kb's block
// counter).  `state` non-NULL: device-selected mode, Kb runs only if its probe does not veto;
// `after_probe` (a cudaEvent_t, may be NULL) is recorded once that decision is final.
int lev_bitvec_launch(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                      const b200lev_opts_t* o, int mode, float mult, int32_t* ref_len,
                      int32_t* hyp_len, int* counter, int32_t* state, int32_t* flags, float* out,
                      int64_t out_si, int Hout, cudaStream_t st, void* after_probe, bool short_form,
                      double* acc) {
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
    a.ref_len = ref_len;
    a.hyp_len = hyp_len;
    a.counter = counter;
    a.state = state;
    a.check_state = state != nullptr;
    a.flags = flags;
    a.slots_log2 = 4;  // buckets of 4 ways: on average at most one token per bucket
    while ((1 << a.slots_log2) < a.R) ++a.slots_log2;
    a.mode = mode;
    a.norm = o->norm;
    a.exclude_last = mode == LEV_MODE_PREFIX ? o->exclude_last : 0;
    a.Hout = Hout;
    a.mult = mult;
    a.padding = (float)o->padding;
    a.out = out;
    a.out_si = out_si;
    a.acc = (short_form && mode == LEV_MODE_FINAL) ? acc : nullptr;
    if (short_form) {  // R <= 64: lane = pair, reference in registers, no tables (lev_bvshort.cu)
        if (getenv("B200LEV_TRACE"))
            fprintf(stderr, "b200lev: short bit-vector kernel, mode %d, R=%d H=%d P=%d\n", mode, a.R, a.H, a.P);
        return lev_bvshort_launch(a, ref->elem_bytes, st);
    }
    if (getenv("B200LEV_TRACE"))
        fprintf(stderr, "b200lev: fused bit-vector kernel, mode %d, R=%d H=%d P=%d W=%d device-selected=%d\n",
                mode, a.R, a.H, a.P, (a.R + 31) / 32, a.check_state);
    return lev_bvfused_launch(a, ref->elem_bytes, st, after_probe);
}
