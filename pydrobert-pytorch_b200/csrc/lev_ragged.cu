// Ragged corpus -> padded batch_first token matrix (bulk-scoring front end, SURVEY 8f #2).
//
// The reference builds its batches on the host, one utterance at a time
// (command_line.py:1110-1121: torch.tensor(transcript + [eos]) per utterance, then
// pad_sequence with padding_value=padding).  Here the corpus lives in HBM as two flat arrays
// (tokens, offsets); row u of the output is utterance sel[u] (or u), then eos, then padding.
// One thread per output element: the stores of a warp are one contiguous segment, the loads
// are contiguous within an utterance (and across utterances when sel is the identity).
#include "lev_common.cuh"

template <typename TT>
__global__ void __launch_bounds__(256)
lev_ragged_kernel(const TT* __restrict__ flat, const int64_t* __restrict__ off,
                  const int64_t* __restrict__ sel, int64_t n, int T, TT eos, TT pad,
                  TT* __restrict__ out) {
    const int64_t total = n * (int64_t)T;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool narrow = total < ((int64_t)1 << 31);
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        int64_t u;
        if (narrow)
            u = (int64_t)((unsigned)idx / (unsigned)T);
        else
            u = idx / T;
        const int64_t j = idx - u * T;
        const int64_t s = sel != nullptr ? sel[u] : u;
        const int64_t b = off[s];
        const int64_t len = off[s + 1] - b;
        out[idx] = j < len ? flat[b + j] : (j == len ? eos : pad);
    }
}

template <typename TT>
static void lev_ragged_launch(const void* flat, const int64_t* off, const int64_t* sel, int64_t n,
                              int64_t T, int64_t eos, int64_t pad, void* out, cudaStream_t st) {
    const int64_t total = n * T;
    int64_t ctas = (total + 255) / 256;
    if (ctas > 148 * 64) ctas = 148 * 64;  // grid-stride beyond 8 resident CTAs x 8 rounds per SM
    lev_launch(lev_ragged_kernel<TT>, dim3((unsigned)ctas), dim3(256), 0, st, (const TT*)flat, off, sel,
               n, (int)T, (TT)eos, (TT)pad, (TT*)out);
}

// b200lev_final_cross, gather path: the cross product's hypotheses as a contiguous sequence-first
// (H, P) tensor of the caller's element width (so wide tokens stay exact).  One thread per pair and
// run of LEV_GATHER_T positions (blockIdx.y): its source column is taken once, the run's loads are
// issued back to back, then stored; the stores of a warp are one contiguous segment per position.
constexpr int LEV_GATHER_T = 8;
template <typename TT>
__global__ void __launch_bounds__(256)
lev_cross_gather_kernel(const TT* __restrict__ hyp, int64_t st, int64_t sn, int H, int AB, int B, int P,
                        TT* __restrict__ out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const TT* __restrict__ src = hyp + (int64_t)(p / AB * B + p % B) * sn;
    TT* __restrict__ dst = out + p;
    for (int t0 = blockIdx.y * LEV_GATHER_T; t0 < H; t0 += gridDim.y * LEV_GATHER_T) {
        TT v[LEV_GATHER_T];
#pragma unroll
        for (int k = 0; k < LEV_GATHER_T; ++k) v[k] = t0 + k < H ? src[(int64_t)(t0 + k) * st] : (TT)0;
#pragma unroll
        for (int k = 0; k < LEV_GATHER_T; ++k)
            if (t0 + k < H) dst[(int64_t)(t0 + k) * P] = v[k];
    }
}

int lev_launch_cross_gather(const b200lev_tokens_t* hyp, int64_t A, int64_t B, int64_t P, void* out,
                            cudaStream_t st) {
    if (P <= 0 || hyp->T <= 0) return B200LEV_OK;
    const int64_t runs = (hyp->T + LEV_GATHER_T - 1) / LEV_GATHER_T;
    const dim3 grid((unsigned)((P + 255) / 256), (unsigned)(runs < 65535 ? runs : 65535)), block(256);
    const int H = (int)hyp->T, AB = (int)(A * B), Bi = (int)B, Pi = (int)P;
#define LEV_GATHER(TT)                                                                                   \
    lev_launch(lev_cross_gather_kernel<TT>, grid, block, 0, st, (const TT*)hyp->data, hyp->stride_t,      \
               hyp->stride_n, H, AB, Bi, Pi, (TT*)out)
    switch (hyp->elem_bytes) {
        case 8: LEV_GATHER(int64_t); break;
        case 4: LEV_GATHER(int32_t); break;
        case 2: LEV_GATHER(int16_t); break;
        default: LEV_GATHER(int8_t); break;
    }
#undef LEV_GATHER
    return lev_check_cuda("lev_cross_gather_kernel");
}

extern "C" int b200lev_ragged_to_padded(const void* flat, int32_t elem_bytes, const int64_t* offsets,
                                        const int64_t* sel, int64_t n, int64_t T, int64_t eos,
                                        int64_t pad, void* out, void* stream) {
    if (n < 0 || T < 1 || T >= ((int64_t)1 << 31)) {
        lev_set_error("ragged_to_padded: n (%lld) must be >= 0 and T (%lld) in [1, 2^31)", (long long)n,
                      (long long)T);
        return B200LEV_ERR_ARG;
    }
    if (elem_bytes != 2 && elem_bytes != 4 && elem_bytes != 8) {
        lev_set_error("ragged_to_padded: elem_bytes (%d) must be 2, 4 or 8", (int)elem_bytes);
        return B200LEV_ERR_ARG;
    }
    if (offsets == nullptr || out == nullptr) {  // flat may be NULL: a corpus of empty utterances
        if (n == 0) return B200LEV_OK;
        lev_set_error("ragged_to_padded: NULL pointer");
        return B200LEV_ERR_ARG;
    }
    if (n == 0) return B200LEV_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (elem_bytes == 2)
        lev_ragged_launch<int16_t>(flat, offsets, sel, n, T, eos, pad, out, st);
    else if (elem_bytes == 4)
        lev_ragged_launch<int32_t>(flat, offsets, sel, n, T, eos, pad, out, st);
    else
        lev_ragged_launch<int64_t>(flat, offsets, sel, n, T, eos, pad, out, st);
    return lev_check_cuda("lev_ragged_kernel");
}
