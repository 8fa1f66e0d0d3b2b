// lev_abi.cu -- the extern "C" boundary declared in include/b200lev.h: argument
// checking, the uniform-cost shortcut (SM:168-174), int/float path selection, workspace
// carving and kernel sequencing.  No device allocation, no host synchronisation.
#include <mutex>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "lev_common.cuh"

static thread_local char g_err[512] = "";

void lev_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int lev_check_cuda(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        lev_set_error("%s: %s", what, cudaGetErrorString(e));
        return B200LEV_ERR_CUDA;
    }
    return B200LEV_OK;
}

// ---- optional per-kernel timing ----------------------------------------------------------
#ifndef B200LEV_EMU
static bool g_prof_on = false;
static cudaEvent_t g_prof_ev[LEV_PROF_NSLOTS][2];
static bool g_prof_used[LEV_PROF_NSLOTS];
static bool g_prof_init = false;
void lev_prof_begin(int slot, cudaStream_t st) {
    if (g_prof_on) cudaEventRecord(g_prof_ev[slot][0], st);
}
void lev_prof_end(int slot, cudaStream_t st) {
    if (g_prof_on) {
        cudaEventRecord(g_prof_ev[slot][1], st);
        g_prof_used[slot] = true;
    }
}
extern "C" int b200lev_profile(int enable) {
    if (enable && !g_prof_init) {
        for (int s = 0; s < LEV_PROF_NSLOTS; ++s)
            for (int k = 0; k < 2; ++k)
                if (cudaEventCreate(&g_prof_ev[s][k]) != cudaSuccess) return lev_check_cuda("cudaEventCreate");
        g_prof_init = true;
    }
    for (int s = 0; s < LEV_PROF_NSLOTS; ++s) g_prof_used[s] = false;
    g_prof_on = enable != 0;
    return B200LEV_OK;
}
extern "C" int b200lev_profile_read(float* ms, int n) {
    for (int s = 0; s < n && s < LEV_PROF_NSLOTS; ++s) {
        ms[s] = -1.0f;
        if (g_prof_init && g_prof_used[s]) {
            if (cudaEventSynchronize(g_prof_ev[s][1]) != cudaSuccess) return lev_check_cuda("cudaEventSynchronize");
            cudaEventElapsedTime(&ms[s], g_prof_ev[s][0], g_prof_ev[s][1]);
        }
    }
    return B200LEV_OK;
}
#else
void lev_prof_begin(int, cudaStream_t) {}
void lev_prof_end(int, cudaStream_t) {}
extern "C" int b200lev_profile(int) { return B200LEV_OK; }
extern "C" int b200lev_profile_read(float* ms, int n) {
    for (int s = 0; s < n; ++s) ms[s] = -1.0f;
    return B200LEV_OK;
}
#endif

extern "C" int b200lev_abi_version(void) { return B200LEV_ABI_VERSION; }
extern "C" const char* b200lev_last_error(void) { return g_err; }

extern "C" int b200lev_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch,
                                    size_t width_bytes, size_t height, int32_t to_device,
                                    void* stream) {
    if (width_bytes == 0 || height == 0) return B200LEV_OK;
    if (dst == nullptr || src == nullptr || dst_pitch < width_bytes || src_pitch < width_bytes) {
        lev_set_error("b200lev_copy2d_async: bad pointers or pitches");
        return B200LEV_ERR_ARG;
    }
#ifdef B200LEV_EMU
    (void)to_device;
    (void)stream;
    for (size_t r = 0; r < height; ++r)
        memcpy((char*)dst + r * dst_pitch, (const char*)src + r * src_pitch, width_bytes);
    return B200LEV_OK;
#else
    cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, height,
                      to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost,
                      (cudaStream_t)stream);
    return lev_check_cuda("cudaMemcpy2DAsync");
#endif
}

extern "C" int b200lev_device_count(void) {
#ifdef B200LEV_EMU
    return 1;
#else
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
#endif
}

static int lev_check_tokens(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                            const b200lev_opts_t* o) {
    if (!ref || !hyp || !o) {
        lev_set_error("NULL argument");
        return B200LEV_ERR_ARG;
    }
    if (ref->T < 0 || hyp->T < 0 || ref->N < 0 || hyp->N < 0) {
        lev_set_error("negative dimension");
        return B200LEV_ERR_ARG;
    }
    if (o->ref_group < 1 || ref->N * o->ref_group != hyp->N) {
        // SM:191-194
        lev_set_error("ref has batch size %lld, but hyp has %lld",
                      (long long)(ref->N * (o->ref_group < 1 ? 1 : o->ref_group)), (long long)hyp->N);
        return B200LEV_ERR_ARG;
    }
    if ((ref->N * ref->T > 0 && !ref->data) || (hyp->N * hyp->T > 0 && !hyp->data)) {
        lev_set_error("NULL token data");
        return B200LEV_ERR_ARG;
    }
    if (ref->T >= (1 << 24) || hyp->T >= (1 << 24) || hyp->N >= ((int64_t)1 << 31)) {
        lev_set_error("dimension too large");
        return B200LEV_ERR_UNSUPPORTED;
    }
    return B200LEV_OK;
}

extern "C" size_t b200lev_workspace_bytes(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                          int32_t kind, int32_t exclude_last) {
    if (!ref || !hyp) return 0;
    return lev_layout(ref, hyp, kind, exclude_last).bytes + 128;
}

static inline char* lev_ws_base(const void* ws) {
    return (char*)(((uintptr_t)ws + 127) & ~(uintptr_t)127);
}

// Fills the cost fields of `p`.  Returns count_mode / float_path through the out-params.
static void lev_classify_costs(const b200lev_opts_t* o, int64_t R, int64_t H, LevParams* p,
                               bool* count_mode, bool* float_path) {
    float ins = o->ins_cost, del = o->del_cost, sub = o->sub_cost;
    float mult = 1.0f;
    bool cm = o->return_mistakes != 0;
    if (ins == del && del == sub && sub > 0.0f) {  // SM:168-174
        if (!cm) mult = ins;
        ins = del = sub = 1.0f;
        cm = false;
    }
    // integer path iff every cost is an integer and every reachable fp32 value of the
    // reference is exact (< 2^24), so int32 arithmetic reproduces it bit for bit
    const float amax = fmaxf(fabsf(ins), fmaxf(fabsf(del), fabsf(sub)));
    const bool integral = floorf(ins) == ins && floorf(del) == del && floorf(sub) == sub &&
                          (double)amax * (double)(R + H + 2) < 16777216.0;
    p->ins_f = ins;
    p->del_f = del;
    p->sub_f = sub;
    p->ins_i = integral ? (int)ins : 0;
    p->del_i = integral ? (int)del : 0;
    p->sub_i = integral ? (int)sub : 0;
    p->mult = mult;
    *count_mode = cm;
    *float_path = !integral;
}

// the fields of `p` every mode shares: workspace tables, the caller's tensors, options, costs
static void lev_params(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                       const b200lev_opts_t* o, const LevLayout& L, char* ws, int32_t* flags,
                       LevParams* p, bool* count_mode, bool* float_path) {
    memset(p, 0, sizeof(*p));
    p->ref_tok = (const int32_t*)(ws + L.off_ref_tok);
    p->hyp_tok = (const int32_t*)(ws + L.off_hyp_tok);
    p->hyp_tok16 = (const uint16_t*)(ws + L.off_hyp_tok16);
    p->Hp16 = L.Hp16;
    p->ref_len = (const int32_t*)(ws + L.off_ref_len);
    p->hyp_len = (const int32_t*)(ws + L.off_hyp_len);
    p->Rp = L.Rp;
    p->Hp = L.Hp;
    p->R = (int)L.R;
    p->H = (int)L.H;
    p->P = (int)L.P;
    p->ref_group = o->ref_group;
    p->norm = o->norm;
    p->exclude_last = o->exclude_last;
    p->padding = (float)o->padding;
    p->flags = flags;
    p->wide_flag = (const int*)(ws + L.off_flags);
    p->ref_raw = ref->data;
    p->hyp_raw = hyp->data;
    p->ref_st = ref->stride_t;
    p->ref_sn = ref->stride_n;
    p->hyp_st = hyp->stride_t;
    p->hyp_sn = hyp->stride_n;
    p->ref_eb = ref->elem_bytes;
    p->hyp_eb = hyp->elem_bytes;
    p->ghist = (int*)(ws + L.off_ghist);
    p->gcursor = (int*)(ws + L.off_gcursor);
    p->gmeta = (int*)(ws + L.off_gmeta);
    p->slots = (int4*)(ws + L.off_slots);
    p->gmeta_order = (int*)(ws + L.off_slots);
    p->nbins = (int)L.nbins;
    p->raw32 = L.off_raw ? (int32_t*)(ws + L.off_raw) : nullptr;
    p->raw16 = (unsigned short*)p->raw32;
    p->Hr = L.Hr;
    p->Hr16 = L.Hr16;
    lev_classify_costs(o, L.R, L.H, p, count_mode, float_path);
}

// What the prologue of a string-matching entry point sets up
struct LevCall {
    LevLayout L;
    char* ws;          // the caller's workspace, aligned
    b200lev_opts_t o;  // the options the call runs with
    LevParams p;
    bool count_mode, float_path;
};

// The argument prologue of the string-matching entry points: checks the token views and the
// options, lays out the workspace for `kind` and checks the caller's buffers.  Returns LEV_EMPTY
// when the call has nothing to write (no pairs, no output rows, or `inner` <= 0), and NULL
// buffers are then fine (only c->L is filled); else B200LEV_OK with *c filled, or an error status
// (`null_status` for a NULL `out` or `ws`).  The call runs with the caller's options after
// `adjust` (may be NULL); the final value and the alignment ignore exclude_last (SM:165).
static constexpr int LEV_EMPTY = 1;
static int lev_begin(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                     const b200lev_opts_t* opts, int kind, const void* out, const void* ws,
                     size_t ws_bytes, int32_t* flags, LevCall* c,
                     void (*adjust)(b200lev_opts_t*) = nullptr, int64_t inner = 1,
                     int null_status = B200LEV_ERR_ARG) {
    const int rc = lev_check_tokens(ref, hyp, opts);
    if (rc) return rc;
    c->o = *opts;
    if (adjust) adjust(&c->o);
    if (kind == B200LEV_WS_FINAL || kind == B200LEV_WS_ALIGN) c->o.exclude_last = 0;
    c->L = lev_layout(ref, hyp, kind, c->o.exclude_last);
    if (hyp->N == 0 || c->L.Hout <= 0 || inner <= 0) return LEV_EMPTY;
    if (!out || !ws) {
        lev_set_error("NULL output or workspace");
        return null_status;
    }
    if (ws_bytes < c->L.bytes + 128) {
        lev_set_error("workspace too small: %zu < %zu", ws_bytes, c->L.bytes + 128);
        return B200LEV_ERR_WORKSPACE;
    }
    c->ws = lev_ws_base(ws);
    lev_params(ref, hyp, &c->o, c->L, c->ws, flags, &c->p, &c->count_mode, &c->float_path);
    return B200LEV_OK;
}

// K0: pack both token tensors into the workspace.  It leaves what the DP kernels need to know
// about the tokens (wider than int32? value range) in 4 state words of the workspace; the
// caller's flags get the same warning bits.  With bv_check the bit-vector launcher has cleared
// the state words before its kernels ran.
static int lev_pack_tokens(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                           const b200lev_opts_t* o, const LevLayout& L, char* ws, int32_t* flags,
                           int bv_check, cudaStream_t st) {
    int32_t* ref_len = (int32_t*)(ws + L.off_ref_len);
    int32_t* state = (int32_t*)(ws + L.off_flags);
    // the group kernel's (class, length) histogram is built by the hypothesis pass whenever the
    // shapes make that kernel eligible (lev_group.cu decides later)
    const int G = lev_group_eligible(L.R, L.H, L.P);
    const size_t clear = sizeof(int32_t) * (size_t)(4 + (G ? L.nbins : 0));
    if (!bv_check && cudaMemsetAsync(state, 0, clear, st) != cudaSuccess) return lev_check_cuda("memset");
    lev_prof_begin(LEV_PROF_PACK_REF, st);
    int rc = lev_launch_pack(ref, o->has_eos, o->eos, o->include_eos, (int32_t*)(ws + L.off_ref_tok),
                             L.Rp, nullptr, 0, ref_len, flags, state, B200LEV_FLAG_REF_NO_EOS, nullptr,
                             1, 0, nullptr, bv_check, st, (int32_t*)(ws + L.off_split_ref));
    lev_prof_end(LEV_PROF_PACK_REF, st);
    if (rc) return rc;
    lev_prof_begin(LEV_PROF_PACK_HYP, st);
    rc = lev_launch_pack(hyp, o->has_eos, o->eos, o->include_eos, (int32_t*)(ws + L.off_hyp_tok), L.Hp,
                         (uint16_t*)(ws + L.off_hyp_tok16), L.Hp16, (int32_t*)(ws + L.off_hyp_len),
                         flags, state, B200LEV_FLAG_HYP_NO_EOS, ref_len, o->ref_group, G,
                         G ? (int*)(ws + L.off_ghist) : nullptr, bv_check, st,
                         (int32_t*)(ws + L.off_split_hyp));
    lev_prof_end(LEV_PROF_PACK_HYP, st);
    return rc;
}

// Device-selected mode forks: once the probe has finished the veto is final, so the wavefront
// path's stand-by chain (seven launches that exit at once when the bit-vector kernel took the
// call) runs on a side stream NEXT TO the bit-vector kernel instead of behind it, and the
// caller's stream joins at the end.  In the vetoed case the bit-vector kernel exits at once and
// the chain does the work.  Nothing the chain touches before its kernels have checked the veto
// overlaps what the bit-vector kernel reads.  One side stream and two events per device, made
// once.  (the side stream and its events are shared by every caller on the device: calls that
// fork are enqueued one at a time)
static std::mutex g_fork_mu;
struct LevFork {
    cudaStream_t side;
    void* after_probe;
    void* joined;
};
#ifndef B200LEV_EMU
static bool lev_fork_get(LevFork* f) {
    static LevFork cache[64];
    static bool have[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return false;
    if (!have[dev]) {
        cudaEvent_t a, b;
        cudaStream_t s2;
        if (cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&a, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&b, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        cache[dev].side = s2;
        cache[dev].after_probe = (void*)a;
        cache[dev].joined = (void*)b;
        have[dev] = true;
    }
    *f = cache[dev];
    return true;
}
// the chain goes to the side stream once the probe is done; returns the stream to use
static cudaStream_t lev_fork_begin(const LevFork& f, bool on) {
    if (!on) return nullptr;
    if (cudaStreamWaitEvent(f.side, (cudaEvent_t)f.after_probe, 0) != cudaSuccess) return nullptr;
    return f.side;
}
static int lev_fork_join(const LevFork& f, cudaStream_t st) {
    if (cudaEventRecord((cudaEvent_t)f.joined, f.side) != cudaSuccess ||
        cudaStreamWaitEvent(st, (cudaEvent_t)f.joined, 0) != cudaSuccess)
        return lev_check_cuda("fork join");
    return B200LEV_OK;
}
#else
static bool lev_fork_get(LevFork*) { return false; }
static cudaStream_t lev_fork_begin(const LevFork&, bool) { return nullptr; }
static int lev_fork_join(const LevFork&, cudaStream_t) { return B200LEV_OK; }
#endif

// b200lev_final / b200lev_final_sums (FINAL; `acc` NULL or the sums) and b200lev_prefix (PREFIX,
// output strides).  Unit costs, short references, sequence-first tensors: the bit-vector path
// (lev_bitvec.cu) takes the whole call -- lengths, warnings and DP -- straight from the raw
// tokens.  Otherwise, or behind its probe when the device selects, K0 and the wavefront DP run.
static int lev_string_match(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                            const b200lev_opts_t* opts, int mode, float* out, int64_t out_si,
                            int64_t out_sn, void* workspace, size_t workspace_bytes,
                            int32_t* flags, double* acc, void* stream) {
    const bool final = mode == LEV_MODE_FINAL;
    LevCall c;
    int rc = lev_begin(ref, hyp, opts, final ? B200LEV_WS_FINAL : B200LEV_WS_PREFIX, out, workspace,
                       workspace_bytes, flags, &c);
    if (rc) return rc == LEV_EMPTY ? B200LEV_OK : rc;
    cudaStream_t st = (cudaStream_t)stream;
    LevParams& p = c.p;
    p.out = out;
    if (!final) {
        p.out_si = out_si;
        p.out_sn = out_sn;
        p.Hout = (int)c.L.Hout;
    }
    std::lock_guard<std::mutex> fork_lock(g_fork_mu);
    const LevBvRoute bv = lev_bitvec_route(ref, hyp, mode, p, c.count_mode, c.float_path);
    LevFork fork;
    const bool forked = bv == LEV_BV_SELECTED && lev_fork_get(&fork);
    if (bv != LEV_BV_NONE) {
        rc = lev_bitvec_launch(bv, ref, hyp, &c.o, mode, c.L, c.ws, p, st, forked ? fork.after_probe : nullptr,
                               acc);
        if (rc) return rc;
    }
    if (bv == LEV_BV_NONE || bv == LEV_BV_SELECTED) {
        cudaStream_t side = lev_fork_begin(fork, forked);
        cudaStream_t cs = side ? side : st;  // the wavefront chain's stream
        p.bv_check = bv == LEV_BV_SELECTED;
        rc = lev_pack_tokens(ref, hyp, &c.o, c.L, c.ws, flags, p.bv_check, cs);
        if (rc == B200LEV_OK) rc = lev_launch_dp(p, mode, c.count_mode, c.float_path, cs);
        if (side) {
            const int jr = lev_fork_join(fork, st);
            if (rc == B200LEV_OK) rc = jr;
        }
    }
    // (Ks accumulates the sums itself)
    if (rc == B200LEV_OK && acc != nullptr && bv != LEV_BV_SHORT)
        rc = lev_launch_err_sum(out, p.ref_len, hyp->N, c.o.ref_group, acc, st);
    return rc;
}

extern "C" int b200lev_final(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                             const b200lev_opts_t* opts, float* out, void* workspace,
                             size_t workspace_bytes, int32_t* flags, void* stream) {
    return lev_string_match(ref, hyp, opts, LEV_MODE_FINAL, out, 0, 0, workspace, workspace_bytes,
                            flags, nullptr, stream);
}

extern "C" int b200lev_final_sums(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                  const b200lev_opts_t* opts, float* out, void* workspace,
                                  size_t workspace_bytes, int32_t* flags, double* acc, void* stream) {
    if (!acc) {
        lev_set_error("NULL accumulator");
        return B200LEV_ERR_ARG;
    }
    if (hyp && hyp->N == 0) return B200LEV_OK;
    return lev_string_match(ref, hyp, opts, LEV_MODE_FINAL, out, 0, 0, workspace, workspace_bytes,
                            flags, acc, stream);
}

// ---- b200lev_final_cross: every reference of a group against every hypothesis of it ------------
// The call is b200lev_final on the expanded pairs p = (g, a, b) -- reference column g*A + a (the
// n-best form, ref_group = B), hypothesis column g*B + b -- without materialising the hypotheses
// where Ks can read them in place: exactly where lev_bitvec_route sends the expanded shape to Ks,
// Ks runs with cross addressing.  Everything else gathers the expanded (H, P) hypotheses into the
// workspace and runs the b200lev_final body on them unchanged.
struct LevCross {
    b200lev_tokens_t hx;  // the expanded hypothesis view (N = P; the data and strides of `hyp`)
    b200lev_opts_t o;     // the caller's options with ref_group = B
    int64_t P;
    bool short_form;      // Ks with cross addressing; else gather + the b200lev_final body
    size_t gather_bytes;  // the gathered hypotheses, 128-byte aligned (0 on the short form)
};

// Checks the arguments of the cross entry points and fills `c`.  B200LEV_OK, or an error status.
static int lev_cross_plan(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp, int64_t A, int64_t B,
                          const b200lev_opts_t* opts, LevCross* c) {
    if (!ref || !hyp || !opts) {
        lev_set_error("NULL argument");
        return B200LEV_ERR_ARG;
    }
    if (A < 0 || B < 0 || ref->N < 0 || hyp->N < 0) {
        lev_set_error("final cross: negative A (%lld), B (%lld) or batch", (long long)A, (long long)B);
        return B200LEV_ERR_ARG;
    }
    if (opts->ref_group != 1) {
        lev_set_error("final cross: ref_group must be 1, got %d", opts->ref_group);
        return B200LEV_ERR_ARG;
    }
    const int64_t G = A > 0 ? ref->N / A : (B > 0 ? hyp->N / B : 0);
    if (ref->N != G * A || (G == 0 ? hyp->N != 0 : (hyp->N % G != 0 || hyp->N / G != B))) {
        lev_set_error("final cross: ref has %lld sequences and hyp %lld, not G*A and G*B for A = %lld, B = %lld",
                      (long long)ref->N, (long long)hyp->N, (long long)A, (long long)B);
        return B200LEV_ERR_ARG;
    }
    const int eb = hyp->elem_bytes;
    if (eb != 1 && eb != 2 && eb != 4 && eb != 8) {
        lev_set_error("unsupported token element size %d", eb);
        return B200LEV_ERR_ARG;
    }
    const int64_t lim = (int64_t)1 << 31;  // (ref->N = G*A and B below 2^31: the product cannot overflow)
    if (G > 0 && (ref->N >= lim || B >= lim || ref->N * B >= lim)) {
        lev_set_error("final cross: G*A*B pairs must be fewer than 2^31");
        return B200LEV_ERR_ARG;
    }
    c->P = G > 0 ? ref->N * B : 0;
    c->hx = *hyp;
    c->hx.N = c->P;
    c->o = *opts;
    c->o.ref_group = B > 0 ? (int32_t)B : 1;
    c->o.exclude_last = 0;
    if (c->P > 0) {  // (before the gather kernel reads anything)
        const int rc = lev_check_tokens(ref, &c->hx, &c->o);
        if (rc) return rc;
    }
    LevParams p;
    memset(&p, 0, sizeof(p));
    bool cm, fp;
    lev_classify_costs(&c->o, ref->T, hyp->T, &p, &cm, &fp);
    p.R = (int)ref->T;
    p.H = (int)hyp->T;
    p.P = (int)c->P;
    p.ref_group = c->o.ref_group;
    c->short_form = c->P > 0 && lev_bitvec_route(ref, &c->hx, LEV_MODE_FINAL, p, cm, fp) == LEV_BV_SHORT;
    c->gather_bytes = c->short_form ? 0 : (size_t)lev_round_up((int64_t)eb * hyp->T * c->P, 128);
    return B200LEV_OK;
}

extern "C" size_t b200lev_final_cross_workspace_bytes(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                                      int64_t A, int64_t B, const b200lev_opts_t* opts) {
    LevCross c;
    if (lev_cross_plan(ref, hyp, A, B, opts, &c) != B200LEV_OK) return 0;
    // the b200lev_final workspace of the expanded shape; the gather path puts the gathered
    // hypotheses in front of it (and aligns both)
    return c.gather_bytes + lev_layout(ref, &c.hx, B200LEV_WS_FINAL, 0).bytes + (c.short_form ? 128 : 256);
}

extern "C" int b200lev_final_cross(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp, int64_t A,
                                   int64_t B, const b200lev_opts_t* opts, float* out, void* workspace,
                                   size_t workspace_bytes, int32_t* flags, void* stream) {
    LevCross c;
    int rc = lev_cross_plan(ref, hyp, A, B, opts, &c);
    if (rc) return rc;
    if (c.P == 0) return B200LEV_OK;
    const bool trace = getenv("B200LEV_TRACE") != nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    if (c.short_form) {
        LevCall k;
        rc = lev_begin(ref, &c.hx, &c.o, B200LEV_WS_FINAL, out, workspace, workspace_bytes, flags, &k);
        if (rc) return rc == LEV_EMPTY ? B200LEV_OK : rc;
        if (trace)
            fprintf(stderr, "b200lev: final cross, short cross form (lev_bv_short_kernel CROSS), A=%lld B=%lld P=%lld\n",
                    (long long)A, (long long)B, (long long)c.P);
        k.p.out = out;
        return lev_bitvec_launch(LEV_BV_SHORT, ref, &c.hx, &k.o, LEV_MODE_FINAL, k.L, k.ws, k.p, st, nullptr,
                                 nullptr, A, B);
    }
    if (!out || !workspace) {
        lev_set_error("NULL output or workspace");
        return B200LEV_ERR_ARG;
    }
    const size_t need = b200lev_final_cross_workspace_bytes(ref, hyp, A, B, opts);
    if (workspace_bytes < need) {
        lev_set_error("workspace too small: %zu < %zu", workspace_bytes, need);
        return B200LEV_ERR_WORKSPACE;
    }
    if (trace)
        fprintf(stderr, "b200lev: final cross, gather + final, A=%lld B=%lld P=%lld\n", (long long)A, (long long)B,
                (long long)c.P);
    char* base = lev_ws_base(workspace);
    rc = lev_launch_cross_gather(hyp, A, B, c.P, base, st);
    if (rc) return rc;
    b200lev_tokens_t hg = c.hx;  // the gathered view: sequence-first, contiguous
    hg.data = base;
    hg.stride_t = c.P;
    hg.stride_n = 1;
    const size_t used = (size_t)(base - (char*)workspace) + c.gather_bytes;
    return lev_string_match(ref, &hg, &c.o, LEV_MODE_FINAL, out, 0, 0, base + c.gather_bytes,
                            workspace_bytes - used, flags, nullptr, stream);
}

extern "C" int b200lev_prefix(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                              const b200lev_opts_t* opts, float* out, int64_t out_stride_i,
                              int64_t out_stride_n, void* workspace, size_t workspace_bytes,
                              int32_t* flags, void* stream) {
    return lev_string_match(ref, hyp, opts, LEV_MODE_PREFIX, out, out_stride_i, out_stride_n,
                            workspace, workspace_bytes, flags, nullptr, stream);
}

// b200lev_error_counts (`counts`) and b200lev_error_alignment (`align`: `ops` with its strides).
// Per pair (C, S, D, I) along the path of error_rate's count mode (SM:292-314; unit costs after
// SM:168-174 take the same cell), or the ops along that path (lev_align.cuh): the alignment keeps
// every cell's choice in the workspace and walks it back.  R <= 64 with one token width: the short
// form, one launch straight from the raw tokens (lev_counts.cuh), where the lane walks its own
// trace.  Otherwise K0 + K1 with the insertion channel, and for the alignment the trace, then one
// thread per pair walks.
static int lev_error_path(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                          const b200lev_opts_t* opts, bool align, int64_t* counts, int8_t* ops,
                          int64_t ops_sk, int64_t ops_sn, void* workspace, size_t workspace_bytes,
                          int32_t* flags, void* stream) {
    const char* what = align ? "error alignment" : "error counts";
    if (opts && opts->ref_group != 1) {
        lev_set_error("%s: ref_group must be 1, got %d", what, opts->ref_group);
        return B200LEV_ERR_ARG;
    }
    LevCall c;
    const int64_t steps = (ref && hyp) ? ref->T + hyp->T : 0;
    int rc = lev_begin(ref, hyp, opts, align ? B200LEV_WS_ALIGN : B200LEV_WS_FINAL,
                       align ? (void*)ops : (void*)counts, workspace, workspace_bytes, flags, &c,
                       [](b200lev_opts_t* o) {
                           o->norm = 0;
                           o->return_mistakes = 1;
                       },
                       align ? steps : 1);
    if (rc) return rc == LEV_EMPTY ? B200LEV_OK : rc;
    cudaStream_t st = (cudaStream_t)stream;
    LevParams& p = c.p;
    if (align) {
        p.trace = (unsigned char*)(c.ws + c.L.off_trace);
        p.trace_pair_bytes = c.L.trace_pair_bytes;
        p.trace_steps = c.L.H + 31;
        p.align_ins = (int*)(c.ws + c.L.off_align_ins);
        p.ops = ops;
        p.ops_sk = ops_sk;
        p.ops_sn = ops_sn;
        p.ops_steps = (int)steps;
    } else {
        p.counts = counts;
    }
    const bool short_form = lev_counts_short_form(ref, hyp);
    if (getenv("B200LEV_TRACE"))
        fprintf(stderr, "b200lev: %s, %s, R=%lld H=%lld P=%lld %s\n", what,
                short_form ? (align ? "lev_counts_short_kernel (trace)" : "lev_counts_short_kernel")
                           : (align ? "pack + lev_warp_kernel (trace) + lev_align_walk_kernel"
                                    : "pack + lev_warp_kernel"),
                (long long)c.L.R, (long long)c.L.H, (long long)c.L.P, c.float_path ? "fp32" : "int32");
    if (short_form) return lev_counts_short_launch(ref, hyp, &c.o, p, c.float_path, st);
    rc = lev_pack_tokens(ref, hyp, &c.o, c.L, c.ws, flags, 0, st);
    if (rc == B200LEV_OK) rc = lev_launch_counts_dp(p, c.float_path, st);
    return rc;
}

extern "C" int b200lev_error_counts(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                    const b200lev_opts_t* opts, int64_t* out, void* workspace,
                                    size_t workspace_bytes, int32_t* flags, void* stream) {
    return lev_error_path(ref, hyp, opts, false, out, nullptr, 0, 0, workspace, workspace_bytes, flags,
                          stream);
}

extern "C" int b200lev_error_alignment(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                       const b200lev_opts_t* opts, int8_t* out, int64_t out_stride_k,
                                       int64_t out_stride_n, void* workspace, size_t workspace_bytes,
                                       int32_t* flags, void* stream) {
    return lev_error_path(ref, hyp, opts, true, nullptr, out, out_stride_k, out_stride_n, workspace,
                          workspace_bytes, flags, stream);
}

// b200lev_infix: per pair the minimum of D[i][r] over the rows of the DP whose column 0 is 0 on every
// row, and with `start` / `end` the match hyp[start:end].  Distance-only calls that the bit-vector
// route sends to Ks run its infix kind straight from the raw tokens; everything else runs K0 + K1 with
// the pinned column (and the start channel for spans).
extern "C" int b200lev_infix(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                             const b200lev_opts_t* opts, float* dist, int64_t* start, int64_t* end,
                             void* workspace, size_t workspace_bytes, int32_t* flags, void* stream) {
    const bool spans = start != nullptr;
    if ((start == nullptr) != (end == nullptr)) {
        lev_set_error("infix: start and end must both be NULL or both be set");
        return B200LEV_ERR_ARG;
    }
    if (opts && opts->ref_group != 1) {
        lev_set_error("infix: ref_group must be 1, got %d", opts->ref_group);
        return B200LEV_ERR_ARG;
    }
    if (opts && spans && opts->norm) {
        lev_set_error("infix: norm applies to distances only, not with start and end");
        return B200LEV_ERR_ARG;
    }
    LevCall c;
    int rc = lev_begin(ref, hyp, opts, B200LEV_WS_FINAL, dist, workspace, workspace_bytes, flags, &c,
                       [](b200lev_opts_t* o) { o->return_mistakes = 0; });
    if (rc) return rc == LEV_EMPTY ? B200LEV_OK : rc;
    cudaStream_t st = (cudaStream_t)stream;
    LevParams& p = c.p;
    p.out = dist;
    p.infix_start = start;
    p.infix_end = end;
    const bool short_form =
        !spans && lev_bitvec_route(ref, hyp, LEV_MODE_FINAL, p, c.count_mode, c.float_path) == LEV_BV_SHORT;
    if (getenv("B200LEV_TRACE"))
        fprintf(stderr, "b200lev: infix, %s, R=%lld H=%lld P=%lld %s\n",
                short_form ? "lev_bv_short_kernel (infix kind)"
                           : (spans ? "pack + lev_warp_kernel (infix, spans)" : "pack + lev_warp_kernel (infix)"),
                (long long)c.L.R, (long long)c.L.H, (long long)c.L.P, c.float_path ? "fp32" : "int32");
    if (short_form)
        return lev_bitvec_launch(LEV_BV_SHORT, ref, hyp, &c.o, LEV_MODE_INFIX, c.L, c.ws, p, st, nullptr, nullptr);
    rc = lev_pack_tokens(ref, hyp, &c.o, c.L, c.ws, flags, 0, st);
    if (rc == B200LEV_OK) rc = lev_launch_infix_dp(p, c.float_path, spans, st);
    return rc;
}

extern "C" int b200lev_completion_count(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                        const b200lev_opts_t* opts, void* workspace,
                                        size_t workspace_bytes, int32_t* umax, int32_t* flags,
                                        void* stream) {
    LevCall c;
    int rc = lev_begin(ref, hyp, opts, B200LEV_WS_COMPLETION, umax, workspace, workspace_bytes, flags, &c,
                       [](b200lev_opts_t* o) {
                           o->return_mistakes = 0;  // SM:479-491: the mask is always taken on the cost row
                           o->norm = 0;
                       });
    if (rc < 0) return rc;
    if (!umax) {  // (an empty batch still writes U = 0)
        lev_set_error("NULL umax");
        return B200LEV_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(umax, 0, sizeof(int32_t), st) != cudaSuccess) return lev_check_cuda("memset");
    if (rc == LEV_EMPTY) return B200LEV_OK;
    const LevLayout& L = c.L;
    LevParams& p = c.p;
    rc = lev_pack_tokens(ref, hyp, &c.o, L, c.ws, flags, 0, st);
    if (rc) return rc;
    int32_t* uid = (int32_t*)(c.ws + L.off_uid);
    int64_t* dtok = (int64_t*)(c.ws + L.off_dtok);
    int32_t* ndist = (int32_t*)(c.ws + L.off_ndist);
    uint32_t* dbits = (uint32_t*)(c.ws + L.off_dbits);
    rc = lev_launch_uid(ref, p.ref_tok, p.wide_flag, p.ref_len, uid, dtok, ndist, L.Rp, st);
    if (rc) return rc;
    if (cudaMemsetAsync(dbits, 0, sizeof(uint32_t) * (size_t)L.Hout * L.P * L.Wd, st) != cudaSuccess)
        return lev_check_cuda("memset");
    p.uid = uid;
    p.ndist = ndist;
    p.dbits = dbits;
    p.Wd = (int)L.Wd;
    p.umax = umax;
    p.Hout = (int)L.Hout;
    return lev_launch_dp(p, LEV_MODE_MASK, false, c.float_path, st);
}

extern "C" int b200lev_completion_fill(const b200lev_tokens_t* ref, const b200lev_tokens_t* hyp,
                                       const b200lev_opts_t* opts, const void* workspace,
                                       size_t workspace_bytes, int64_t U, int64_t* out,
                                       int64_t out_stride_i, int64_t out_stride_n, void* stream) {
    // (a NULL output counts as a bad workspace here)
    LevCall c;
    const int rc = lev_begin(ref, hyp, opts, B200LEV_WS_COMPLETION, out, workspace, workspace_bytes,
                             nullptr, &c, nullptr, U, B200LEV_ERR_WORKSPACE);
    if (rc) return rc == LEV_EMPTY ? B200LEV_OK : rc;
    const LevLayout& L = c.L;
    return lev_launch_completion_fill((const uint32_t*)(c.ws + L.off_dbits),
                                      (const int64_t*)(c.ws + L.off_dtok), (const int*)(c.ws + L.off_flags), L.Rp,
                                      L.Hout, L.P, L.Wd,
                                      opts->ref_group, U, opts->padding, out, out_stride_i,
                                      out_stride_n, (cudaStream_t)stream);
}
