// lev_loss.cu -- K5 (OCD loss), K6 (MWER epilogue), K7 (bulk error sums), the
// fill_after_eos scan and the INT32 issue-rate microbenchmark.
//
// "SM" = src/pydrobert/torch/_string.py of the reference.
#include "lev_common.cuh"

// ---- element loaders / storers ---------------------------------------------------------
template <int DT> struct LevElem;
template <> struct LevElem<B200LEV_F32> {
    typedef float T; typedef float Acc;
    static __device__ __forceinline__ float ld(const float* p) { return *p; }
    static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
    static __device__ __forceinline__ float round(float v) { return v; }
};
template <> struct LevElem<B200LEV_F64> {
    typedef double T; typedef double Acc;
    static __device__ __forceinline__ double ld(const double* p) { return *p; }
    static __device__ __forceinline__ void st(double* p, double v) { *p = v; }
    static __device__ __forceinline__ double round(double v) { return v; }
};
template <> struct LevElem<B200LEV_F16> {
    typedef __half T; typedef float Acc;
    static __device__ __forceinline__ float ld(const __half* p) { return __half2float(*p); }
    static __device__ __forceinline__ void st(__half* p, float v) { *p = __float2half(v); }
    static __device__ __forceinline__ float round(float v) { return __half2float(__float2half(v)); }
};
template <> struct LevElem<B200LEV_BF16> {
    typedef __nv_bfloat16 T; typedef float Acc;
    static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16(v); }
    static __device__ __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16(v)); }
};

template <typename A> __device__ __forceinline__ A lev_exp(A x);
template <> __device__ __forceinline__ float lev_exp<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ double lev_exp<double>(double x) { return exp(x); }
template <typename A> __device__ __forceinline__ A lev_log(A x);
template <> __device__ __forceinline__ float lev_log<float>(float x) { return logf(x); }
template <> __device__ __forceinline__ double lev_log<double>(double x) { return log(x); }

template <typename A>
__device__ __forceinline__ A lev_warp_sum(A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(LEV_FULL_MASK, v, o);
    return v;
}
template <typename A>
__device__ __forceinline__ A lev_warp_max(A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const A t = __shfl_xor_sync(LEV_FULL_MASK, v, o);
        v = t > v ? t : v;
    }
    return v;
}

// ======================= K5: hard OCD loss (SM:1229-1251) ==============================
// One warp per (a, b) row of V logits.  per = (1/|S|) * sum_{t in S} w_t (lse - z_t).
template <int DT>
__global__ void __launch_bounds__(256)
lev_ocd_fwd_kernel(const typename LevElem<DT>::T* __restrict__ logits, int64_t rows, int64_t B,
                   int64_t V, int64_t ls_a, int64_t ls_b, const int64_t* __restrict__ targets,
                   int64_t U, int64_t ts_a, int64_t ts_b,
                   const typename LevElem<DT>::Acc* __restrict__ weight, int64_t ignore_index,
                   typename LevElem<DT>::Acc* __restrict__ per,
                   typename LevElem<DT>::Acc* __restrict__ lse_out, int32_t* __restrict__ flags) {
    typedef typename LevElem<DT>::Acc A;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int64_t a = row / B, b = row - a * B;
    const typename LevElem<DT>::T* z = logits + a * ls_a + b * ls_b;
    A mx = -(A)INFINITY;
    for (int64_t v = lane; v < V; v += 32) {
        const A x = (A)LevElem<DT>::ld(z + v);
        mx = x > mx ? x : mx;
    }
    mx = lev_warp_max(mx);
    if (!(mx > -(A)INFINITY && mx < (A)INFINITY)) mx = (A)0;
    A se = (A)0;
    for (int64_t v = lane; v < V; v += 32) se += lev_exp<A>((A)LevElem<DT>::ld(z + v) - mx);
    se = lev_warp_sum(se);
    const A lse = mx + lev_log<A>(se);
    const int64_t* tg = targets + a * ts_a + b * ts_b;
    A acc = (A)0;
    int cnt = 0;
    for (int64_t u = lane; u < U; u += 32) {
        const int64_t t = tg[u];
        if (t == ignore_index) continue;
        if (t < 0 || t >= V) {  // not a class: reported (the reference raises), never read
            if (flags) atomicOr(flags, B200LEV_FLAG_BAD_TARGET);
            continue;
        }
        const A w = weight ? weight[t] : (A)1;
        acc += w * (lse - (A)LevElem<DT>::ld(z + t));  // SM:1232-1238
        cnt += 1;
    }
    acc = lev_warp_sum(acc);
    cnt = lev_warp_sum(cnt);
    if (lane == 0) {
        per[row] = acc / (A)(cnt > 1 ? cnt : 1);  // SM:1239-1241
        lse_out[row] = lse;
    }
}

// mean (SM:1242-1246): mean over sequences of (sum over steps / #steps with targets);
// sum (SM:1247-1248).  Single CTA, fixed summation order (deterministic): blocks of 32
// sequences on the lanes (coalesced when the sequence axis is the inner one), the 32 warps
// take every 32nd step (four loads in flight each: the kernel is pure load latency), warp 0
// adds the 32 partials of each sequence in order.
template <typename A>
__global__ void __launch_bounds__(1024)
lev_ocd_reduce_kernel(const A* __restrict__ per, int64_t Adim, int64_t Bdim,
                      const int64_t* __restrict__ targets, int64_t U, int64_t ts_a, int64_t ts_b,
                      int64_t ignore_index, int reduction, int seq_axis, A* __restrict__ denom,
                      A* __restrict__ loss) {
    __shared__ A psum[32][32];
    __shared__ int phave[32][32];
    __shared__ A part[1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t nseq = seq_axis == 0 ? Bdim : Adim;   // number of sequences
    const int64_t nstep = seq_axis == 0 ? Adim : Bdim;  // steps per sequence
    A acc = (A)0;  // (warp 0 only) this lane's sequences, in order
    for (int64_t q0 = 0; q0 < nseq; q0 += 32) {
        const int64_t q = q0 + lane;
        A s = (A)0;
        int have = 0;
        if (q < nseq)
            for (int64_t t0 = warp; t0 < nstep; t0 += 128) {
                A v[4];
                int64_t g[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int64_t t = t0 + 32 * k;
                    const bool in = t < nstep;
                    const int64_t a = seq_axis == 0 ? t : q, b = seq_axis == 0 ? q : t;
                    v[k] = in ? per[a * Bdim + b] : (A)0;
                    g[k] = (in && U > 0) ? targets[a * ts_a + b * ts_b] : ignore_index;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    s += v[k];
                    have += g[k] != ignore_index;
                }
            }
        psum[warp][lane] = s;
        phave[warp][lane] = have;
        __syncthreads();
        if (warp == 0 && q < nseq) {
            A tot = (A)0;
            int h = 0;
            for (int w = 0; w < 32; ++w) {
                tot += psum[w][lane];
                h += phave[w][lane];
            }
            const A d = (A)(h > 1 ? h : 1);
            denom[q] = d;
            acc += (reduction == B200LEV_REDUCE_MEAN) ? tot / d : tot;
        }
        __syncthreads();
    }
    if (warp == 0) {
        acc = lev_warp_sum(acc);
        if (lane == 0) part[0] = acc;
    }
    __syncthreads();
    if (tid == 0) loss[0] = (reduction == B200LEV_REDUCE_MEAN) ? part[0] / (A)nseq : part[0];
}

// d per / d z_v = coef * softmax_v - [v in S] w_v / |S|,  coef = sum_t w_t / |S|
template <int DT>
__global__ void __launch_bounds__(256)
lev_ocd_bwd_kernel(const typename LevElem<DT>::T* __restrict__ logits, int64_t rows, int64_t B,
                   int64_t V, int64_t ls_a, int64_t ls_b, const int64_t* __restrict__ targets,
                   int64_t U, int64_t ts_a, int64_t ts_b,
                   const typename LevElem<DT>::Acc* __restrict__ weight, int64_t ignore_index,
                   int reduction, int seq_axis, int64_t nseq,
                   const typename LevElem<DT>::Acc* __restrict__ lse_in,
                   const typename LevElem<DT>::Acc* __restrict__ denom,
                   const typename LevElem<DT>::Acc* __restrict__ grad_out,
                   typename LevElem<DT>::T* __restrict__ grad) {
    typedef typename LevElem<DT>::Acc A;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int64_t a = row / B, b = row - a * B;
    const typename LevElem<DT>::T* z = logits + a * ls_a + b * ls_b;
    typename LevElem<DT>::T* g = grad + row * V;
    A go;
    if (reduction == B200LEV_REDUCE_NONE)
        go = grad_out[row];
    else if (reduction == B200LEV_REDUCE_SUM)
        go = grad_out[0];
    else
        go = grad_out[0] / (denom[seq_axis == 0 ? b : a] * (A)nseq);
    const int64_t* tg = targets + a * ts_a + b * ts_b;
    A wsum = (A)0;
    int cnt = 0;
    for (int64_t u = lane; u < U; u += 32) {
        const int64_t t = tg[u];
        if (t != ignore_index && t >= 0 && t < V) {  // the forward reports the others
            wsum += weight ? weight[t] : (A)1;
            cnt += 1;
        }
    }
    wsum = lev_warp_sum(wsum);
    cnt = lev_warp_sum(cnt);
    const A inv = (A)1 / (A)(cnt > 1 ? cnt : 1);
    const A coef = go * wsum * inv;
    const A lse = lse_in[row];
    for (int64_t v = lane; v < V; v += 32)
        LevElem<DT>::st(g + v, coef * lev_exp<A>((A)LevElem<DT>::ld(z + v) - lse));
    __syncwarp();
    // the targets of one row are distinct (sorted-unique), so these stores do not collide
    for (int64_t u = lane; u < U; u += 32) {
        const int64_t t = tg[u];
        if (t != ignore_index && t >= 0 && t < V) {
            const A w = weight ? weight[t] : (A)1;
            LevElem<DT>::st(g + t, coef * lev_exp<A>((A)LevElem<DT>::ld(z + t) - lse) - go * w * inv);
        }
    }
}

template <int DT>
static int lev_ocd_forward_t(const void* logits, int64_t A_, int64_t B, int64_t V, int64_t ls_a,
                             int64_t ls_b, const int64_t* targets, int64_t U, int64_t ts_a,
                             int64_t ts_b, const void* weight, int64_t ignore_index,
                             int reduction, int seq_axis, void* per, void* lse, void* denom,
                             void* loss, int32_t* flags, cudaStream_t st) {
    typedef typename LevElem<DT>::Acc A;
    const int64_t rows = A_ * B;
    if (rows > 0) {
        dim3 block(256), grid((unsigned)((rows + 7) / 8));
        lev_launch(lev_ocd_fwd_kernel<DT>, grid, block, 0, st,
                   (const typename LevElem<DT>::T*)logits, rows, B, V, ls_a, ls_b, targets, U, ts_a,
                   ts_b, (const A*)weight, ignore_index, (A*)per, (A*)lse, flags);
    }
    if (reduction != B200LEV_REDUCE_NONE)
        lev_launch(lev_ocd_reduce_kernel<A>, dim3(1), dim3(1024), 0, st, (const A*)per, A_, B, targets,
                   U, ts_a, ts_b, ignore_index, reduction, seq_axis, (A*)denom, (A*)loss);
    return lev_check_cuda("lev_ocd_fwd_kernel");
}

template <int DT>
static int lev_ocd_backward_t(const void* logits, int64_t A_, int64_t B, int64_t V, int64_t ls_a,
                              int64_t ls_b, const int64_t* targets, int64_t U, int64_t ts_a,
                              int64_t ts_b, const void* weight, int64_t ignore_index,
                              int reduction, int seq_axis, const void* lse, const void* denom,
                              const void* grad_out, void* grad, cudaStream_t st) {
    typedef typename LevElem<DT>::Acc A;
    const int64_t rows = A_ * B;
    if (rows <= 0) return B200LEV_OK;
    dim3 block(256), grid((unsigned)((rows + 7) / 8));
    lev_launch(lev_ocd_bwd_kernel<DT>, grid, block, 0, st, (const typename LevElem<DT>::T*)logits,
               rows, B, V, ls_a, ls_b, targets, U, ts_a, ts_b, (const A*)weight, ignore_index, reduction,
               seq_axis, seq_axis == 0 ? B : A_, (const A*)lse, (const A*)denom, (const A*)grad_out,
               (typename LevElem<DT>::T*)grad);
    return lev_check_cuda("lev_ocd_bwd_kernel");
}

#define LEV_DT_SWITCH(dtype, CALL)                                        \
    switch (dtype) {                                                      \
        case B200LEV_F32: return CALL(B200LEV_F32);                       \
        case B200LEV_F16: return CALL(B200LEV_F16);                       \
        case B200LEV_BF16: return CALL(B200LEV_BF16);                     \
        case B200LEV_F64: return CALL(B200LEV_F64);                       \
        default:                                                          \
            lev_set_error("unsupported floating dtype code %d", (int)dtype); \
            return B200LEV_ERR_ARG;                                       \
    }

extern "C" int b200lev_ocd_forward(const void* logits, int32_t dtype, int64_t A, int64_t B,
                                   int64_t V, int64_t ls_a, int64_t ls_b, const int64_t* targets,
                                   int64_t U, int64_t ts_a, int64_t ts_b, const void* weight,
                                   int64_t ignore_index, int32_t reduction, int32_t seq_axis,
                                   void* per, void* lse, void* denom, void* loss, int32_t* flags,
                                   void* stream) {
#define CALL(DT)                                                                                  \
    lev_ocd_forward_t<DT>(logits, A, B, V, ls_a, ls_b, targets, U, ts_a, ts_b, weight,            \
                          ignore_index, reduction, seq_axis, per, lse, denom, loss, flags,        \
                          (cudaStream_t)stream)
    LEV_DT_SWITCH(dtype, CALL)
#undef CALL
}

extern "C" int b200lev_ocd_backward(const void* logits, int32_t dtype, int64_t A, int64_t B,
                                    int64_t V, int64_t ls_a, int64_t ls_b, const int64_t* targets,
                                    int64_t U, int64_t ts_a, int64_t ts_b, const void* weight,
                                    int64_t ignore_index, int32_t reduction, int32_t seq_axis,
                                    const void* lse, const void* denom, const void* grad_out,
                                    void* grad_logits, void* stream) {
#define CALL(DT)                                                                                  \
    lev_ocd_backward_t<DT>(logits, A, B, V, ls_a, ls_b, targets, U, ts_a, ts_b, weight,           \
                           ignore_index, reduction, seq_axis, lse, denom, grad_out, grad_logits,  \
                           (cudaStream_t)stream)
    LEV_DT_SWITCH(dtype, CALL)
#undef CALL
}

// ======================= K6: MWER epilogue (SM:1463-1471) ==============================
// One warp per n-best group: e = er - mean_m(er) (if sub_avg), p = softmax(log_probs),
// per = e * p.  p is rounded to the dtype of log_probs first, as torch's softmax
// output is (bf16/fp16 inputs), then the product is taken in fp32 (fp64 for fp64).
template <int DT>
__global__ void __launch_bounds__(256)
lev_mwer_fwd_kernel(const float* __restrict__ er, const typename LevElem<DT>::T* __restrict__ lp,
                    int64_t N, int64_t M, int64_t sn, int64_t sm, int sub_avg,
                    typename LevElem<DT>::Acc* __restrict__ per) {
    typedef typename LevElem<DT>::Acc A;
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (n >= N) return;
    float es = 0.f;
    A mx = -(A)INFINITY;
    for (int64_t m = lane; m < M; m += 32) {
        es += er[n * M + m];
        const A x = (A)LevElem<DT>::ld(lp + n * sn + m * sm);
        mx = x > mx ? x : mx;
    }
    es = lev_warp_sum(es);
    mx = lev_warp_max(mx);
    const float mean = sub_avg ? es / (float)M : 0.f;  // SM:1463-1464
    A se = (A)0;
    for (int64_t m = lane; m < M; m += 32) se += lev_exp<A>((A)LevElem<DT>::ld(lp + n * sn + m * sm) - mx);
    se = lev_warp_sum(se);
    for (int64_t m = lane; m < M; m += 32) {
        const A p = LevElem<DT>::round(lev_exp<A>((A)LevElem<DT>::ld(lp + n * sn + m * sm) - mx) / se);
        per[n * M + m] = (A)(er[n * M + m] - mean) * p;  // SM:1465
    }
}

// d/dlp_m sum_k go_k e_k p_k = p_m (go_m e_m - sum_k p_k go_k e_k)
template <int DT>
__global__ void __launch_bounds__(256)
lev_mwer_bwd_kernel(const float* __restrict__ er, const typename LevElem<DT>::T* __restrict__ lp,
                    int64_t N, int64_t M, int64_t sn, int64_t sm, int sub_avg, int reduction,
                    const typename LevElem<DT>::Acc* __restrict__ grad_out,
                    typename LevElem<DT>::T* __restrict__ grad) {
    typedef typename LevElem<DT>::Acc A;
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (n >= N) return;
    float es = 0.f;
    A mx = -(A)INFINITY;
    for (int64_t m = lane; m < M; m += 32) {
        es += er[n * M + m];
        const A x = (A)LevElem<DT>::ld(lp + n * sn + m * sm);
        mx = x > mx ? x : mx;
    }
    es = lev_warp_sum(es);
    mx = lev_warp_max(mx);
    const float mean = sub_avg ? es / (float)M : 0.f;
    A se = (A)0;
    for (int64_t m = lane; m < M; m += 32) se += lev_exp<A>((A)LevElem<DT>::ld(lp + n * sn + m * sm) - mx);
    se = lev_warp_sum(se);
    A dot = (A)0;
    for (int64_t m = lane; m < M; m += 32) {
        const A p = lev_exp<A>((A)LevElem<DT>::ld(lp + n * sn + m * sm) - mx) / se;
        A go = reduction == B200LEV_REDUCE_NONE ? grad_out[n * M + m] : grad_out[0];
        if (reduction == B200LEV_REDUCE_MEAN) go = go / (A)(N * M);
        dot += p * go * (A)(er[n * M + m] - mean);
    }
    dot = lev_warp_sum(dot);
    for (int64_t m = lane; m < M; m += 32) {
        const A p = lev_exp<A>((A)LevElem<DT>::ld(lp + n * sn + m * sm) - mx) / se;
        A go = reduction == B200LEV_REDUCE_NONE ? grad_out[n * M + m] : grad_out[0];
        if (reduction == B200LEV_REDUCE_MEAN) go = go / (A)(N * M);
        LevElem<DT>::st(grad + n * M + m, p * (go * (A)(er[n * M + m] - mean) - dot));
    }
}

// deterministic single-CTA sum / mean of n values
template <typename A>
__global__ void __launch_bounds__(256)
lev_reduce_kernel(const A* __restrict__ x, int64_t n, int mean, A* __restrict__ out) {
    __shared__ A part[256];
    const int tid = threadIdx.x;
    A acc = (A)0;
    for (int64_t i = tid; i < n; i += 256) acc += x[i];
    part[tid] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) part[tid] += part[tid + o];
        __syncthreads();
    }
    if (tid == 0) out[0] = mean ? part[0] / (A)(n > 0 ? n : 1) : part[0];
}

template <int DT>
static int lev_mwer_forward_t(const float* er, const void* lp, int64_t N, int64_t M, int64_t sn,
                              int64_t sm, int sub_avg, int reduction, void* per, void* loss,
                              cudaStream_t st) {
    typedef typename LevElem<DT>::Acc A;
    if (N > 0 && M > 0)
        lev_launch(lev_mwer_fwd_kernel<DT>, dim3((unsigned)((N + 7) / 8)), dim3(256), 0, st, er,
                   (const typename LevElem<DT>::T*)lp, N, M, sn, sm, sub_avg, (A*)per);
    if (reduction != B200LEV_REDUCE_NONE)
        lev_launch(lev_reduce_kernel<A>, dim3(1), dim3(256), 0, st, (const A*)per, N * M,
                   reduction == B200LEV_REDUCE_MEAN ? 1 : 0, (A*)loss);
    return lev_check_cuda("lev_mwer_fwd_kernel");
}

template <int DT>
static int lev_mwer_backward_t(const float* er, const void* lp, int64_t N, int64_t M, int64_t sn,
                               int64_t sm, int sub_avg, int reduction, const void* grad_out,
                               void* grad, cudaStream_t st) {
    typedef typename LevElem<DT>::Acc A;
    if (N <= 0 || M <= 0) return B200LEV_OK;
    lev_launch(lev_mwer_bwd_kernel<DT>, dim3((unsigned)((N + 7) / 8)), dim3(256), 0, st, er,
               (const typename LevElem<DT>::T*)lp, N, M, sn, sm, sub_avg, reduction,
               (const A*)grad_out, (typename LevElem<DT>::T*)grad);
    return lev_check_cuda("lev_mwer_bwd_kernel");
}

extern "C" int b200lev_mwer_forward(const float* er, const void* log_probs, int32_t dtype,
                                    int64_t N, int64_t M, int64_t lp_sn, int64_t lp_sm,
                                    int32_t sub_avg, int32_t reduction, void* per, void* loss,
                                    void* stream) {
#define CALL(DT)                                                                             \
    lev_mwer_forward_t<DT>(er, log_probs, N, M, lp_sn, lp_sm, sub_avg, reduction, per, loss, \
                           (cudaStream_t)stream)
    LEV_DT_SWITCH(dtype, CALL)
#undef CALL
}

extern "C" int b200lev_mwer_backward(const float* er, const void* log_probs, int32_t dtype,
                                     int64_t N, int64_t M, int64_t lp_sn, int64_t lp_sm,
                                     int32_t sub_avg, int32_t reduction, const void* grad_out,
                                     void* grad, void* stream) {
#define CALL(DT)                                                                                \
    lev_mwer_backward_t<DT>(er, log_probs, N, M, lp_sn, lp_sm, sub_avg, reduction, grad_out,    \
                            grad, (cudaStream_t)stream)
    LEV_DT_SWITCH(dtype, CALL)
#undef CALL
}

// ======================= minimum-Bayes-risk epilogue ===================================
// One warp per group, next to K6 and with its softmax: p = softmax(log_probs[n]) rounded to the
// dtype of log_probs, risk[n, i] = sum_a p_a * er[n, a, i] in the accumulation type, rounded to
// the dtype of log_probs, best[n] = its arg min.  Lane l sums column i = i0 + l over a = 0 .. M-1
// in that order, p_a broadcast from the lane that computed it: every column is summed in the same
// order, so identical hypotheses get bitwise identical risks, and equal risks go to the lowest i.
template <int DT>
__global__ void __launch_bounds__(256)
lev_mbr_kernel(const float* __restrict__ er, const typename LevElem<DT>::T* __restrict__ lp, int64_t N,
               int64_t M, int64_t sn, int64_t sm, typename LevElem<DT>::T* __restrict__ risk,
               int64_t* __restrict__ best) {
    typedef typename LevElem<DT>::Acc A;
    const int lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (n >= N) return;
    const typename LevElem<DT>::T* row = lp + n * sn;
    A mx = -(A)INFINITY;
    for (int64_t m = lane; m < M; m += 32) {
        const A x = (A)LevElem<DT>::ld(row + m * sm);
        mx = x > mx ? x : mx;
    }
    mx = lev_warp_max(mx);
    A se = (A)0;
    for (int64_t m = lane; m < M; m += 32) se += lev_exp<A>((A)LevElem<DT>::ld(row + m * sm) - mx);
    se = lev_warp_sum(se);
    const float* __restrict__ e = er + n * M * M;
    A bv = (A)INFINITY;
    int64_t bi = M;  // (no finite risk: 0 below)
    for (int64_t i0 = 0; i0 < M; i0 += 32) {
        const int64_t i = i0 + lane;
        A acc = (A)0;
        for (int64_t a0 = 0; a0 < M; a0 += 32) {
            const int64_t am = a0 + lane;
            const A pm = am < M ? LevElem<DT>::round(lev_exp<A>((A)LevElem<DT>::ld(row + am * sm) - mx) / se) : (A)0;
            const int kn = M - a0 < 32 ? (int)(M - a0) : 32;
            for (int k = 0; k < kn; ++k) {
                const A pa = __shfl_sync(LEV_FULL_MASK, pm, k);
                if (i < M) acc += pa * (A)e[(a0 + k) * M + i];
            }
        }
        if (i < M) {
            const A r = LevElem<DT>::round(acc);
            LevElem<DT>::st(risk + n * M + i, r);
            if (r < bv) {
                bv = r;
                bi = i;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const A ov = __shfl_xor_sync(LEV_FULL_MASK, bv, o);
        const int64_t oi = __shfl_xor_sync(LEV_FULL_MASK, bi, o);
        if (ov < bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    if (lane == 0) best[n] = bi < M ? bi : 0;
}

template <int DT>
static int lev_mbr_t(const float* er, const void* lp, int64_t N, int64_t M, int64_t sn, int64_t sm, void* risk,
                     int64_t* best, cudaStream_t st) {
    lev_launch(lev_mbr_kernel<DT>, dim3((unsigned)((N + 7) / 8)), dim3(256), 0, st, er,
               (const typename LevElem<DT>::T*)lp, N, M, sn, sm, (typename LevElem<DT>::T*)risk, best);
    return lev_check_cuda("lev_mbr_kernel");
}

extern "C" int b200lev_mbr(const float* er, const void* log_probs, int32_t dtype, int64_t N, int64_t M,
                           int64_t lp_sn, int64_t lp_sm, void* risk, int64_t* best, void* stream) {
    if (N < 0 || M < 0 || (N > 0 && M < 1)) {
        lev_set_error("mbr: need N >= 0 and M >= 1, got N = %lld, M = %lld", (long long)N, (long long)M);
        return B200LEV_ERR_ARG;
    }
    if (N == 0) return B200LEV_OK;
    if (!er || !log_probs || !risk || !best) {
        lev_set_error("mbr: NULL pointer");
        return B200LEV_ERR_ARG;
    }
    if (N >= ((int64_t)1 << 34)) {  // (grid of N / 8 CTAs)
        lev_set_error("mbr: too many groups");
        return B200LEV_ERR_UNSUPPORTED;
    }
#define CALL(DT) lev_mbr_t<DT>(er, log_probs, N, M, lp_sn, lp_sm, risk, best, (cudaStream_t)stream)
    LEV_DT_SWITCH(dtype, CALL)
#undef CALL
}

// ======================= K7: bulk error sums ===========================================
// command_line.py:1135-1147 accumulates per-utterance .item()s on the host; here the
// three totals stay on the device in fp64 (exact for integer error counts) so that a
// multi-GPU job needs a single 24-byte all-reduce.
__global__ void __launch_bounds__(256)
lev_err_sum_kernel(const float* __restrict__ er, const int32_t* __restrict__ ref_lens, int64_t P,
                   int ref_group, double* __restrict__ acc) {
    __shared__ double s_er[256];
    __shared__ double s_len[256];
    const int tid = threadIdx.x;
    double e = 0.0, l = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * 256 + tid; i < P; i += (int64_t)gridDim.x * 256) {
        e += (double)er[i];
        l += (double)ref_lens[i / ref_group];
    }
    s_er[tid] = e;
    s_len[tid] = l;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) {
            s_er[tid] += s_er[tid + o];
            s_len[tid] += s_len[tid + o];
        }
        __syncthreads();
    }
    if (tid == 0) {
        atomicAdd(acc + 0, s_er[0]);
        atomicAdd(acc + 1, s_len[0]);
        if (blockIdx.x == 0) atomicAdd(acc + 2, (double)P);
    }
}

int lev_launch_err_sum(const float* er, const int32_t* ref_lens, int64_t P, int ref_group,
                       double* acc, cudaStream_t st) {
    int64_t blocks = (P + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    lev_prof_begin(LEV_PROF_ERR_SUM, st);
    lev_launch(lev_err_sum_kernel, dim3((unsigned)blocks), dim3(256), 0, st, er, ref_lens, P,
               ref_group, acc);
    lev_prof_end(LEV_PROF_ERR_SUM, st);
    return lev_check_cuda("lev_err_sum_kernel");
}

// ======================= fill_after_eos scan (SM:30-42) =================================
// mask[o, t, i] = 1 iff some t' < t has tokens[o, t', i] == eos  (strictly after the first
// eos).  The broadcasted fill itself (SM:42) is a masked_fill on the caller's side.
__global__ void __launch_bounds__(256)
lev_after_eos_kernel(const int64_t* __restrict__ tok, int64_t outer, int64_t T, int64_t inner,
                     int64_t eos, unsigned char* __restrict__ mask) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= outer * inner) return;
    const int64_t o = idx / inner, i = idx - o * inner;
    const int64_t base = o * T * inner + i;
    unsigned char seen = 0;
    for (int64_t t = 0; t < T; ++t) {
        mask[base + t * inner] = seen;
        if (tok[base + t * inner] == eos) seen = 1;
    }
}

extern "C" int b200lev_after_eos_mask(const int64_t* tokens, int64_t outer, int64_t T,
                                      int64_t inner, int64_t eos, unsigned char* mask,
                                      void* stream) {
    const int64_t n = outer * inner;
    if (n <= 0 || T <= 0) return B200LEV_OK;
    lev_launch(lev_after_eos_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0,
               (cudaStream_t)stream, tokens, outer, T, inner, eos, mask);
    return lev_check_cuda("lev_after_eos_kernel");
}

// ======================= INT32 issue-rate microbenchmark ================================
// Roofline denominator for the DP kernels (bench.py): 8 independent chains per thread.
//   variant 0: IADD3        x = x + y
//   variant 1: VIMNMX       x = min(x, y) (with a perturbation so it cannot fold)
//   variant 2: VIADDMNMX    x = min(x + a, y)
//   variant 3: the 4-instruction DP cell (ISETP, predicated IADD, 2x VIADDMNMX)
template <int VAR>
__global__ void __launch_bounds__(256) lev_int32_peak_kernel(int iters, int a, int b, int* sink) {
    int x[8], y[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        x[q] = (int)threadIdx.x + q * a;
        y[q] = (int)blockIdx.x + q * b;
    }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (VAR == 0) {
                x[q] = x[q] + y[q];
                y[q] = y[q] + x[q];
            } else if (VAR == 1) {
                x[q] = min(x[q], y[q] ^ it);
                y[q] = max(y[q], x[q] ^ a);
            } else if (VAR == 2) {
                x[q] = __viaddmin_s32(x[q], a, y[q]);
                y[q] = __viaddmax_s32(y[q], b, x[q]);
            } else {
                const int sb = y[q] + ((x[q] != it) ? a : 0);
                const int t = __viaddmin_s32(x[q], b, sb);
                y[q] = __viaddmin_s32(y[q], a, t);
                x[q] = t;
            }
        }
    }
    int acc = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) acc ^= x[q] ^ y[q];
    if (acc == 0x7fffffff) sink[0] = acc;
}

extern "C" int b200lev_int32_peak_kernel(int32_t variant, int64_t blocks, int64_t iters,
                                         int32_t* sink, double* ops, void* stream) {
    dim3 grid((unsigned)blocks), block(256);
    cudaStream_t st = (cudaStream_t)stream;
    double per_iter = 0;
    switch (variant) {
        case 0: lev_launch(lev_int32_peak_kernel<0>, grid, block, 0, st, (int)iters, 3, 5, sink); per_iter = 16; break;
        case 1: lev_launch(lev_int32_peak_kernel<1>, grid, block, 0, st, (int)iters, 3, 5, sink); per_iter = 32; break;
        case 2: lev_launch(lev_int32_peak_kernel<2>, grid, block, 0, st, (int)iters, 3, 5, sink); per_iter = 16; break;
        case 3: lev_launch(lev_int32_peak_kernel<3>, grid, block, 0, st, (int)iters, 3, 5, sink); per_iter = 32; break;
        default:
            lev_set_error("unknown microbenchmark variant %d", (int)variant);
            return B200LEV_ERR_ARG;
    }
    if (ops) *ops = per_iter * (double)iters * (double)blocks * 256.0;
    return lev_check_cuda("lev_int32_peak_kernel");
}
