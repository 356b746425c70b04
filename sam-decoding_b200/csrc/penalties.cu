// Repetition, presence and frequency penalties on the draft rows: samd_apply_penalties (include/samd_b200.h).
//
// Row j of request b predicts the token after prompt + emitted tokens + the draft tokens on the path from node 0 to
// node j.  With c[t] = occurrences of t in (emitted + path) and seen[t] = t in the prompt or c[t] > 0, every seen entry
// becomes, in fp32 with each operation rounded on its own (no FMA contraction), then rounded once into the logits dtype:
//     x = x < 0 ? x * r : x / r;   x = x - f * c[t];   x = x - p * (c[t] > 0)
// The per-slot state is a dense count table [S][V]: bits 0..30 the output count, bit 31 "seen in the prompt".
//
// One CTA per (request, PEN_CHUNK vocabulary entries), for all the request's rows.  It
//   1. reads the path table once: node j's owner is the first (path, depth) entry listing it (its path from node 0 is the
//      owner path's prefix; a node on no live path is not penalized), and the node tokens that fall in the chunk form
//      the path-token set (a bitmap plus a list of distinct tokens);
//   2. reads its chunk of the count row with 16-byte loads, once, and compacts the nonzero entries that are not path
//      tokens into shared memory in vocabulary order (a block scan);
//   3. applies the history-only entries to every live row with c = the count, and every (row, path token) pair with
//      c = count + the token's multiplicity on that row's path.
// So every (row, token) is rewritten at most once, each from its own inputs: the results do not depend on the chunking,
// the batch or graph / eager execution.
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <limits.h>

#define PEN_THREADS 256
#define PEN_PER_THREAD 8                        // count entries per thread: two 16-byte loads
#define PEN_CHUNK (PEN_THREADS * PEN_PER_THREAD)
#define PEN_MAX_NODES 256
#define PEN_PROMPT 0x80000000u

namespace {

template <int kDtype> struct Elem;
template <> struct Elem<SAMD_DTYPE_FP32> {
    using T = float;
    static __device__ __forceinline__ float load(const T *p) { return *p; }
    static __device__ __forceinline__ void store(T *p, float x) { *p = x; }
};
template <> struct Elem<SAMD_DTYPE_BF16> {
    using T = __nv_bfloat16;
    static __device__ __forceinline__ float load(const T *p) { return __bfloat162float(*p); }
    static __device__ __forceinline__ void store(T *p, float x) { *p = __float2bfloat16_rn(x); }
};
template <> struct Elem<SAMD_DTYPE_FP16> {
    using T = __half;
    static __device__ __forceinline__ float load(const T *p) { return __half2float(*p); }
    static __device__ __forceinline__ void store(T *p, float x) { *p = __float2half_rn(x); }
};

// a seen entry with output count c (-inf stays -inf, NaN stays NaN)
__device__ __forceinline__ float penalize(float x, int c, float r, float p, float f) {
    x = x < 0.f ? __fmul_rn(x, r) : __fdiv_rn(x, r);
    x = __fsub_rn(x, __fmul_rn(f, (float)c));
    return __fsub_rn(x, __fmul_rn(p, c > 0 ? 1.f : 0.f));
}

template <int kDtype>
__global__ void __launch_bounds__(PEN_THREADS) apply_penalties_kernel(samd_penalty_args A) {
    using E = Elem<kDtype>;
    using T = typename E::T;
    __shared__ int s_owner[PEN_MAX_NODES];      // first path-table entry p * D + d listing node j; INT_MAX: none
    __shared__ int s_parent[PEN_MAX_NODES];
    __shared__ int s_tok[PEN_MAX_NODES];
    __shared__ int s_path_tok[PEN_MAX_NODES];   // distinct node tokens in [lo, hi)
    __shared__ uint32_t s_on_path[PEN_CHUNK / 32];
    __shared__ int s_hist_tok[PEN_CHUNK];       // history-only entries of the chunk: token, count word
    __shared__ uint32_t s_hist_word[PEN_CHUNK];
    __shared__ int s_warp[PEN_THREADS / 32];
    __shared__ int s_n_path;

    const int b = blockIdx.y, tid = threadIdx.x, V = A.vocab, Tn = A.n_nodes;
    const int lo = blockIdx.x * PEN_CHUNK, hi = min(lo + PEN_CHUNK, V);
    if (A.done_dev && A.done_dev[b]) return;
    const int s = A.slots_dev ? A.slots_dev[b] : b;
    if (s < 0 || s >= A.n_slots) return;
    const float r = A.repetition_dev[s], pp = A.presence_dev[s], ff = A.frequency_dev[s];
    if (r == 1.f && pp == 0.f && ff == 0.f) return;                        // neutral: not touched
    const int n = min(Tn, A.n_nodes_dev ? A.n_nodes_dev[b] : Tn);
    if (n <= 0) return;
    const bool has_path = A.tokens_dev != nullptr, table = has_path && A.retrieve_dev != nullptr;

    // 1. owners, parents and the chunk's path tokens
    for (int j = tid; j < n; j += PEN_THREADS) {
        s_owner[j] = table ? INT_MAX : j;
        s_parent[j] = j - 1;                                               // identity chain
        s_tok[j] = has_path ? A.tokens_dev[(size_t)b * Tn + j] : -1;
    }
    for (int w = tid; w < PEN_CHUNK / 32; w += PEN_THREADS) s_on_path[w] = 0;
    if (tid == 0) s_n_path = 0;
    __syncthreads();
    if (table) {
        const int P = A.n_paths, D = A.depth;
        const int np = min(P, A.n_paths_dev ? A.n_paths_dev[b] : P);
        const int32_t *ret = A.retrieve_dev + (size_t)b * P * D;
        for (int p = tid; p < np; p += PEN_THREADS)
            for (int d = 0; d < D; ++d) {
                const int j = ret[p * D + d];
                if (j < 0) break;                                          // -1: the end of the path
                if (j < n) atomicMin(&s_owner[j], p * D + d);
            }
        __syncthreads();
        for (int j = tid; j < n; j += PEN_THREADS) {
            const int o = s_owner[j];
            s_parent[j] = (o == INT_MAX || o % D == 0) ? -1 : ret[o - 1];
        }
    }
    if (has_path)
        for (int j = tid; j < n; j += PEN_THREADS) {
            const int t = s_tok[j];
            if (s_owner[j] == INT_MAX || t < lo || t >= hi) continue;
            const uint32_t bit = 1u << ((t - lo) & 31);
            if (!(atomicOr(&s_on_path[(t - lo) >> 5], bit) & bit)) s_path_tok[atomicAdd(&s_n_path, 1)] = t;
        }
    __syncthreads();

    // 2. the chunk of the count row, once; nonzero entries that are not path tokens, compacted in vocabulary order
    const uint32_t *crow = reinterpret_cast<const uint32_t *>(A.counts_dev) + (size_t)s * V;
    const int k0 = lo + tid * PEN_PER_THREAD;
    uint32_t v[PEN_PER_THREAD];
    if ((reinterpret_cast<uintptr_t>(crow) & 15) == 0 && k0 + PEN_PER_THREAD <= hi) {
        const uint4 x = *reinterpret_cast<const uint4 *>(crow + k0), y = *reinterpret_cast<const uint4 *>(crow + k0 + 4);
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    } else {
#pragma unroll
        for (int e = 0; e < PEN_PER_THREAD; ++e) v[e] = k0 + e < hi ? crow[k0 + e] : 0u;
    }
    int mine = 0;
#pragma unroll
    for (int e = 0; e < PEN_PER_THREAD; ++e) {
        const int o = k0 + e - lo;
        if (v[e] && (s_on_path[o >> 5] >> (o & 31) & 1u)) v[e] = 0;
        mine += v[e] != 0;
    }
    int incl = mine;                                                       // block exclusive scan of `mine`
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(SAMD_FULL, incl, o);
        if ((tid & 31) >= o) incl += y;
    }
    if ((tid & 31) == 31) s_warp[tid >> 5] = incl;
    __syncthreads();
    int at = incl - mine, n_hist = 0;
    for (int w = 0; w < PEN_THREADS / 32; ++w) {
        if (w < (tid >> 5)) at += s_warp[w];
        n_hist += s_warp[w];
    }
#pragma unroll
    for (int e = 0; e < PEN_PER_THREAD; ++e)
        if (v[e]) {
            s_hist_tok[at] = k0 + e;
            s_hist_word[at++] = v[e];
        }
    __syncthreads();

    // 3. the rewrites: history-only tokens on every live row, then every (row, path token) pair
    T *L = reinterpret_cast<T *>(A.logits_dev) + (size_t)b * A.batch_stride;
    for (int q = tid; q < n_hist * n; q += PEN_THREADS) {
        const int j = q / n_hist, e = q - j * n_hist;
        if (s_owner[j] == INT_MAX) continue;
        T *x = L + (size_t)j * A.row_stride + s_hist_tok[e];
        E::store(x, penalize(E::load(x), (int)(s_hist_word[e] & ~PEN_PROMPT), r, pp, ff));
    }
    const int n_path = s_n_path;
    for (int q = tid; q < n_path * n; q += PEN_THREADS) {
        const int j = q / n_path, t = s_path_tok[q - j * n_path];
        if (s_owner[j] == INT_MAX) continue;
        int m = 0;
        for (int k = j, g = 0; k >= 0 && k < n && g < n; k = s_parent[k], ++g) m += s_tok[k] == t;
        const uint32_t w = crow[t];
        const int c = (int)(w & ~PEN_PROMPT) + m;
        if (c == 0 && !(w & PEN_PROMPT)) continue;
        T *x = L + (size_t)j * A.row_stride + t;
        E::store(x, penalize(E::load(x), c, r, pp, ff));
    }
}

template <int kDtype>
void launch(const samd_penalty_args &a, cudaStream_t stream) {
    const dim3 grid((a.vocab + PEN_CHUNK - 1) / PEN_CHUNK, a.batch);
    apply_penalties_kernel<kDtype><<<grid, PEN_THREADS, 0, stream>>>(a);
}

}  // namespace

extern "C" int samd_apply_penalties(const samd_penalty_args *a, void *stream) {
    SAMD_REQUIRE(a && a->logits_dev && a->counts_dev && a->repetition_dev && a->presence_dev && a->frequency_dev,
                 "samd_apply_penalties: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->batch <= 65535 && a->vocab > 0 && a->n_slots > 0, "samd_apply_penalties: bad shape");
    SAMD_REQUIRE(a->n_nodes > 0 && a->n_nodes <= PEN_MAX_NODES, "samd_apply_penalties: n_nodes must be in [1, 256]");
    SAMD_REQUIRE(!a->retrieve_dev || (a->tokens_dev && a->n_paths > 0 && a->depth > 0),
                 "samd_apply_penalties: a path table needs the node tokens and a positive shape");
    SAMD_REQUIRE(a->dtype == SAMD_DTYPE_BF16 || a->dtype == SAMD_DTYPE_FP16 || a->dtype == SAMD_DTYPE_FP32,
                 "samd_apply_penalties: bad dtype");
    if (a->dtype == SAMD_DTYPE_BF16) launch<SAMD_DTYPE_BF16>(*a, (cudaStream_t)stream);
    else if (a->dtype == SAMD_DTYPE_FP16) launch<SAMD_DTYPE_FP16>(*a, (cudaStream_t)stream);
    else launch<SAMD_DTYPE_FP32>(*a, (cudaStream_t)stream);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
