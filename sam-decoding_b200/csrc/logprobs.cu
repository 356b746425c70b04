// Per-token log-probabilities of the accepted path: samd_token_logprobs (include/samd_b200.h).
//
// After a verify launch, position j < count[b] of request b was predicted by logits row r = indices[b][j] (-1: the
// request's last live row, as samd_verify_compact reads it), and the token it predicted is tokens[b][j + 1], or
// next_token[b] for the last position.  The value is the raw log_softmax(float32(row))[target], with no temperature and
// no top-p / top-k, plus optionally the n_top best (value descending, index ascending, NaN largest: oracle.row_topk).
//
// One CTA per (position, request); positions past count, and finished requests, exit at once, so only the scored rows
// are read from DRAM, each exactly once.  A thread owns the 16-byte chunks c = tid + k * LP_THREADS of its row and
// keeps an online (max, sum of exp) pair and, with n_top, its own eight best keys.  The chunk -> thread map and every
// reduction order depend only on V and the block size, not on where the row sits: a row that is not 16-byte aligned is
// read with element loads of the same chunks, so the same row gives bit-identical results at any (b, j), B, or alignment.
// The aligned path issues its LP_UNROLL loads ahead of a __syncwarp, so that ptxas cannot interleave them with the
// arithmetic (it did, to save registers: one load in flight per thread).
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#define LP_THREADS 512
#define LP_UNROLL 8             // 16-byte loads in flight per thread
#define LP_MAX_TOP 8

namespace {

__device__ __forceinline__ uint32_t lp_skey(float f) {       // order-preserving key (NaN largest, +0 == -0)
    const uint32_t b = __float_as_uint(f), a = b & 0x7FFFFFFFu;
    if (a > 0x7F800000u) return 0xFFFFFFFFu;
    if (a == 0) return 0x80000000u;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float lp_key_float(uint32_t k) {  // inverse of lp_skey (NaN for the NaN key)
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

template <int kDtype> struct Chunk;                            // one 16-byte chunk: E elements
template <> struct Chunk<SAMD_DTYPE_FP32> { static constexpr int E = 4; using T = float; };
template <> struct Chunk<SAMD_DTYPE_BF16> { static constexpr int E = 8; using T = __nv_bfloat16; };
template <> struct Chunk<SAMD_DTYPE_FP16> { static constexpr int E = 8; using T = __half; };

template <int kDtype>
__device__ __forceinline__ float to_f(typename Chunk<kDtype>::T v) {
    if constexpr (kDtype == SAMD_DTYPE_FP32) return v;
    else if constexpr (kDtype == SAMD_DTYPE_BF16) return __bfloat162float(v);
    else return __half2float(v);
}

template <int kDtype>
__device__ __forceinline__ void unpack(const uint4 &u, float *x) {
    using T = typename Chunk<kDtype>::T;
    const T *e = reinterpret_cast<const T *>(&u);
#pragma unroll
    for (int i = 0; i < Chunk<kDtype>::E; ++i) x[i] = to_f<kDtype>(e[i]);
}

// chunk c of a row with element loads (-inf past V): an unaligned row, or the partial last chunk
template <int kDtype>
__device__ __forceinline__ void load_chunk(const typename Chunk<kDtype>::T *row, int c, int V, float *x) {
    constexpr int E = Chunk<kDtype>::E;
#pragma unroll
    for (int i = 0; i < E; ++i) x[i] = c * E + i < V ? to_f<kDtype>(row[c * E + i]) : -INFINITY;
}

// (m, s): running maximum and sum of exp(x - m).  A -inf adds nothing; a NaN makes s NaN (torch.log_softmax's NaN row).
// Rescales use expf: their errors compound, while the per-element __expf errors are independent.
__device__ __forceinline__ void merge_ms(float &m, float &s, float m2, float s2) {
    const float M = fmaxf(m, m2);
    if (M == -INFINITY) {
        s += s2;
        return;
    }
    s = (s == 0.f ? 0.f : s * expf(m - M)) + (s2 == 0.f ? 0.f : s2 * expf(m2 - M));
    m = M;
}

__device__ __forceinline__ void top_insert(unsigned long long (&L)[LP_MAX_TOP], unsigned long long k) {
    if (k <= L[LP_MAX_TOP - 1]) return;
    L[LP_MAX_TOP - 1] = k;
#pragma unroll
    for (int q = LP_MAX_TOP - 1; q > 0; --q)
        if (L[q] > L[q - 1]) {
            const unsigned long long t = L[q];
            L[q] = L[q - 1];
            L[q - 1] = t;
        }
}

__device__ __forceinline__ unsigned long long block_max_u64(unsigned long long v, unsigned long long *s_red) {
    for (int o = 16; o; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(SAMD_FULL, v, o);
        v = w > v ? w : v;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long t = s_red[0];
    for (int w = 1; w < LP_THREADS / 32; ++w) t = s_red[w] > t ? s_red[w] : t;
    return t;
}

template <int kDtype, bool kTop>
__global__ void __launch_bounds__(LP_THREADS) token_logprobs_kernel(samd_logprob_args A) {
    using T = typename Chunk<kDtype>::T;
    constexpr int E = Chunk<kDtype>::E;
    __shared__ float s_m[LP_THREADS / 32], s_s[LP_THREADS / 32];
    __shared__ unsigned long long s_red[LP_THREADS / 32];
    const int j = blockIdx.x, b = blockIdx.y, W = A.width;
    if (A.done_dev && A.done_dev[b]) return;
    const int a = min(A.count_dev[b], W);
    if (j >= a) return;
    const int n_rows = max(1, min(A.n_nodes, A.n_nodes_dev ? A.n_nodes_dev[b] : A.n_nodes));
    int r = A.indices_dev ? A.indices_dev[(size_t)b * W + j] : j;
    if (r < 0 || r >= n_rows) r = n_rows - 1;                   // -1 wraps to the request's last live row
    const bool last = j + 1 >= a;
    const int target = last ? A.next_token_dev[b] : (A.tokens_dev ? A.tokens_dev[(size_t)b * W + j + 1] : -1);
    const int V = A.vocab;
    const T *row = reinterpret_cast<const T *>(A.logits_dev) + (size_t)b * A.batch_stride + (size_t)r * A.row_stride;
    const int n_chunks = (V + E - 1) / E;

    float m = -INFINITY, s = 0.f;
    unsigned long long L[LP_MAX_TOP];
#pragma unroll
    for (int q = 0; q < LP_MAX_TOP; ++q) L[q] = 0ull;
    auto take = [&](const float *x, int c) {
        float vm = x[0];
#pragma unroll
        for (int i = 1; i < E; ++i) vm = fmaxf(vm, x[i]);
        if (vm > m) {
            s *= expf(m - vm);                                  // (m = -inf: s is 0); rare, so the accurate expf
            m = vm;
        }
#pragma unroll
        for (int i = 0; i < E; ++i) {
            s += x[i] == -INFINITY ? 0.f : __expf(x[i] - m);
            if (kTop && c * E + i < V)
                top_insert(L, ((unsigned long long)lp_skey(x[i]) << 32) | (0xFFFFFFFFu - (uint32_t)(c * E + i)));
        }
    };
    int c = threadIdx.x;
    if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {        // aligned: LP_UNROLL 16-byte loads issued back to back
        const uint4 *rv = reinterpret_cast<const uint4 *>(row);
        for (const int n_full = V / E; c + (LP_UNROLL - 1) * LP_THREADS < n_full; c += LP_UNROLL * LP_THREADS) {
            uint4 u[LP_UNROLL];
#pragma unroll
            for (int k = 0; k < LP_UNROLL; ++k) u[k] = rv[c + k * LP_THREADS];
            __syncwarp();                                       // (coherent loads do not move past it)
#pragma unroll
            for (int k = 0; k < LP_UNROLL; ++k) {
                float x[E];
                unpack<kDtype>(u[k], x);
                take(x, c + k * LP_THREADS);
            }
        }
    }
    for (; c < n_chunks; c += LP_THREADS) {                     // the rest, in the same chunk order
        float x[E];
        load_chunk<kDtype>(row, c, V, x);
        take(x, c);
    }

    // (m, s) over the block: a fixed shuffle tree, then the warps in order
    for (int o = 16; o; o >>= 1) {
        const float m2 = __shfl_xor_sync(SAMD_FULL, m, o), s2 = __shfl_xor_sync(SAMD_FULL, s, o);
        merge_ms(m, s, m2, s2);
    }
    if ((threadIdx.x & 31) == 0) {
        s_m[threadIdx.x >> 5] = m;
        s_s[threadIdx.x >> 5] = s;
    }
    __syncthreads();
    m = s_m[0];
    s = s_s[0];
    for (int w = 1; w < LP_THREADS / 32; ++w) merge_ms(m, s, s_m[w], s_s[w]);
    const float log_s = logf(s);

    if (threadIdx.x == 0) {
        const float lp = target >= 0 && target < V ? (to_f<kDtype>(row[target]) - m) - log_s : __int_as_float(0x7FC00000);
        if (last) A.out_next_logprob_dev[b] = lp;
        else A.out_logprob_dev[(size_t)b * W + j] = lp;
    }
    if (kTop) {
        int32_t *ids = last ? A.out_next_top_ids_dev + (size_t)b * A.n_top : A.out_top_ids_dev + ((size_t)b * W + j) * A.n_top;
        float *lps = last ? A.out_next_top_logprob_dev + (size_t)b * A.n_top
                          : A.out_top_logprob_dev + ((size_t)b * W + j) * A.n_top;
        for (int q = 0; q < A.n_top; ++q) {                     // n_top rounds: the best head, its owner pops it
            const unsigned long long best = block_max_u64(L[0], s_red);
            if (L[0] == best) {
#pragma unroll
                for (int p = 0; p + 1 < LP_MAX_TOP; ++p) L[p] = L[p + 1];
                L[LP_MAX_TOP - 1] = 0ull;
            }
            if (threadIdx.x == 0) {
                ids[q] = (int32_t)(0xFFFFFFFFu - (uint32_t)best);
                lps[q] = (lp_key_float((uint32_t)(best >> 32)) - m) - log_s;
            }
        }
    }
}

template <int kDtype>
void launch(const samd_logprob_args &a, cudaStream_t stream) {
    const dim3 grid(a.width, a.batch);
    if (a.n_top > 0) token_logprobs_kernel<kDtype, true><<<grid, LP_THREADS, 0, stream>>>(a);
    else token_logprobs_kernel<kDtype, false><<<grid, LP_THREADS, 0, stream>>>(a);
}

}  // namespace

extern "C" int samd_token_logprobs(const samd_logprob_args *a, void *stream) {
    SAMD_REQUIRE(a && a->logits_dev && a->count_dev && a->next_token_dev && a->out_next_logprob_dev,
                 "samd_token_logprobs: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->n_nodes > 0 && a->vocab > 0 && a->width > 0 && a->batch <= 65535,
                 "samd_token_logprobs: bad shape");
    SAMD_REQUIRE(a->indices_dev || a->width <= a->n_nodes, "samd_token_logprobs: identity path wider than n_nodes");
    SAMD_REQUIRE(a->dtype == SAMD_DTYPE_BF16 || a->dtype == SAMD_DTYPE_FP16 || a->dtype == SAMD_DTYPE_FP32,
                 "samd_token_logprobs: bad dtype");
    SAMD_REQUIRE(a->n_top >= 0 && a->n_top <= LP_MAX_TOP && a->n_top <= a->vocab, "samd_token_logprobs: n_top must be in [0, 8]");
    SAMD_REQUIRE(a->width == 1 || a->out_logprob_dev, "samd_token_logprobs: out_logprob_dev is NULL");
    SAMD_REQUIRE(a->n_top == 0 || (a->out_next_top_ids_dev && a->out_next_top_logprob_dev &&
                                   (a->width == 1 || (a->out_top_ids_dev && a->out_top_logprob_dev))),
                 "samd_token_logprobs: n_top > 0 needs the top-n outputs");
    if (a->dtype == SAMD_DTYPE_BF16) launch<SAMD_DTYPE_BF16>(*a, (cudaStream_t)stream);
    else if (a->dtype == SAMD_DTYPE_FP16) launch<SAMD_DTYPE_FP16>(*a, (cudaStream_t)stream);
    else launch<SAMD_DTYPE_FP32>(*a, (cudaStream_t)stream);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
