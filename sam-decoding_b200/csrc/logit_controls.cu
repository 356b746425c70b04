// Logit bias, banned token sequences and min_tokens on the draft rows: samd_apply_logit_controls (include/samd_b200.h).
//
// Row j of request b predicts output position hist_len + depth(j) + 1 from its own context: the output so far, then the
// node tokens on the path from node 0 to node j (the admission form has no node tokens and predicts hist_len).  The
// slot's tables say what to do with it:
//     bias     x = round_to_dtype(fp32(x) + bias) for each (distinct) biased id; a -inf bias stores -inf
//     bans     -inf on the last id of every bad word whose head ends the context, and, before min_tokens, on EOS and on
//              the last id of every stop sequence whose head ends the context
//
// One CTA per request.  It
//   1. stages the node tokens, each node's owner (the first (path, depth) entry listing it; a node on no live path is not
//      touched), the last CTX history tokens and the slot's tables in shared memory;
//   2. builds every live row's context tail, CTX tokens right-aligned: its owner path backwards from node j, then the
//      history (never before output position 0);
//   3. phase A, the (row, bias entry) pairs: each (row, token) is read-modify-written once, because the ids are distinct;
//   4. phase B, after a barrier, the (row, sequence) pairs of the bans: these only store the constant -inf, so the order
//      in which threads reach a token does not matter.
// The results depend only on the inputs, not on the launch shape or on graph / eager execution.  The work is sparse: at
// most SAMD_BIAS_MAX + SAMD_BAD_MAX_SEQS + SAMD_STOP_MAX_SEQS + 1 entries per row and no pass over the vocabulary.
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <limits.h>
#include <math.h>

#define CTL_THREADS 256
#define CTL_MAX_NODES 256
#define CTX (SAMD_BAD_MAX_LEN - 1)                 // context tokens a sequence's head can read
#define CTL_PAIRS (SAMD_BAD_MAX_SEQS + SAMD_STOP_MAX_SEQS + 1)

static_assert(SAMD_STOP_MAX_LEN == SAMD_BAD_MAX_LEN, "stops and bad words share the context tail");

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

template <int kDtype>
__global__ void __launch_bounds__(CTL_THREADS) logit_controls_kernel(samd_logit_control_args A) {
    using E = Elem<kDtype>;
    using T = typename E::T;
    __shared__ int s_owner[CTL_MAX_NODES];          // first path-table entry p * D + d listing node j; INT_MAX: none
    __shared__ int s_tok[CTL_MAX_NODES];
    __shared__ int s_ctx[CTL_MAX_NODES][CTX];       // each live row's context tail, right-aligned
    __shared__ int s_ctx_n[CTL_MAX_NODES];          // its valid tokens (-1: the row is not touched)
    __shared__ int s_pos[CTL_MAX_NODES];            // the output position it predicts
    __shared__ int s_hist[CTX];
    __shared__ int s_bias_id[SAMD_BIAS_MAX];
    __shared__ float s_bias[SAMD_BIAS_MAX];
    __shared__ int s_bad[SAMD_BAD_MAX_SEQS * SAMD_BAD_MAX_LEN];
    __shared__ int s_stop[SAMD_STOP_MAX_SEQS * SAMD_STOP_MAX_LEN];
    __shared__ int s_bad_len[SAMD_BAD_MAX_SEQS];
    __shared__ int s_stop_len[SAMD_STOP_MAX_SEQS];

    const int b = blockIdx.x, tid = threadIdx.x, V = A.vocab, Tn = A.n_nodes;
    if (A.done_dev && A.done_dev[b]) return;
    const int s = A.slots_dev ? A.slots_dev[b] : b;
    if (s < 0 || s >= A.n_slots) return;
    const int n = min(Tn, A.n_nodes_dev ? A.n_nodes_dev[b] : Tn);
    if (n <= 0) return;
    const int n_bias = min(max(A.bias_n_dev[s], 0), SAMD_BIAS_MAX), m = A.min_tokens_dev[s];
    const bool has_path = A.tokens_dev != nullptr, table = has_path && A.retrieve_dev != nullptr;
    const bool has_stop = A.stop_tokens_dev != nullptr && A.stop_len_dev != nullptr;
    const int hl = A.hist_len_dev ? min(max(A.hist_len_dev[s], 0), A.hist_stride) : 0;
    const int h = min(hl, CTX);                     // history tokens staged: output positions hl - h .. hl - 1

    // 1. the slot's tables, the history tail, node tokens and owners
    if (tid < SAMD_BAD_MAX_SEQS) {
        s_bad_len[tid] = A.bad_len_dev[(size_t)s * SAMD_BAD_MAX_SEQS + tid];
        s_stop_len[tid] = has_stop ? A.stop_len_dev[(size_t)s * SAMD_STOP_MAX_SEQS + tid] : 0;
    }
    for (int k = tid; k < SAMD_BAD_MAX_SEQS * SAMD_BAD_MAX_LEN; k += CTL_THREADS) {
        s_bad[k] = A.bad_tokens_dev[(size_t)s * SAMD_BAD_MAX_SEQS * SAMD_BAD_MAX_LEN + k];
        s_stop[k] = has_stop ? A.stop_tokens_dev[(size_t)s * SAMD_STOP_MAX_SEQS * SAMD_STOP_MAX_LEN + k] : -1;
    }
    for (int e = tid; e < n_bias; e += CTL_THREADS) {
        s_bias_id[e] = A.bias_ids_dev[(size_t)s * SAMD_BIAS_MAX + e];
        s_bias[e] = A.bias_dev[(size_t)s * SAMD_BIAS_MAX + e];
    }
    if (tid < h) s_hist[tid] = A.hist_dev[(size_t)s * A.hist_stride + hl - h + tid];
    for (int j = tid; j < Tn; j += CTL_THREADS) {
        s_owner[j] = table ? INT_MAX : j;
        s_tok[j] = has_path ? A.tokens_dev[(size_t)b * Tn + j] : -1;
    }
    __syncthreads();
    bool active = n_bias > 0;                       // block-uniform: every thread reads the same shared values
    for (int k = 0; k < SAMD_BAD_MAX_SEQS; ++k) active |= s_bad_len[k] > 0;
    if (m > 0) {
        bool any_stop = false;
        for (int k = 0; k < SAMD_STOP_MAX_SEQS; ++k) any_stop |= s_stop_len[k] > 0;
        active |= (A.eos_token >= 0 && A.eos_token < V) || any_stop;
    }
    if (!active) return;                            // neutral: not touched
    const int P = A.n_paths, D = A.depth;
    const int32_t *ret = table ? A.retrieve_dev + (size_t)b * P * D : nullptr;
    if (table) {
        const int np = min(P, A.n_paths_dev ? A.n_paths_dev[b] : P);
        for (int p = tid; p < np; p += CTL_THREADS)
            for (int d = 0; d < D; ++d) {
                const int j = ret[p * D + d];
                if (j < 0) break;                   // -1: the end of the path
                if (j < n) atomicMin(&s_owner[j], p * D + d);
            }
        __syncthreads();
    }

    // 2. every live row's context tail: its path backwards from node j (the owner entry's prefix), then the history
    for (int j = tid; j < n; j += CTL_THREADS) {
        const int o = s_owner[j];
        if (o == INT_MAX) { s_ctx_n[j] = -1; continue; }
        const int d = !has_path ? -1 : table ? o % D : j;      // depth; -1: no node tokens
        const int n_ctx = min(CTX, hl + d + 1);
        int node = d, at = h - 1;                               // next path entry backwards, next history token
        for (int i = CTX - 1; i >= CTX - n_ctx; --i) {
            int t;
            if (node >= 0) {
                const int k = table ? ret[o - (d - node)] : node;
                t = (k >= 0 && k < Tn) ? s_tok[k] : -1;
                --node;
            } else {
                t = s_hist[at--];
            }
            s_ctx[j][i] = t;
        }
        s_ctx_n[j] = n_ctx;
        s_pos[j] = hl + d + 1;
    }
    __syncthreads();

    // 3. phase A: the bias, one read-modify-write per (row, entry)
    T *L = reinterpret_cast<T *>(A.logits_dev) + (size_t)b * A.batch_stride;
    for (int q = tid; q < n * n_bias; q += CTL_THREADS) {
        const int j = q / n_bias, e = q - j * n_bias;
        const int t = s_bias_id[e];
        if (s_ctx_n[j] < 0 || t < 0 || t >= V) continue;
        T *x = L + (size_t)j * A.row_stride + t;
        const float bias = s_bias[e];
        E::store(x, bias == -INFINITY ? -INFINITY : __fadd_rn(E::load(x), bias));
    }
    __syncthreads();                                            // (phase B's -inf lands after any bias)

    // 4. phase B: bad words on every row; EOS and stop sequences on rows before min_tokens
    for (int q = tid; q < n * CTL_PAIRS; q += CTL_THREADS) {
        const int j = q / CTL_PAIRS, k = q - j * CTL_PAIRS;
        const int n_ctx = s_ctx_n[j];
        if (n_ctx < 0) continue;
        const bool early = s_pos[j] < m;
        T *row = L + (size_t)j * A.row_stride;
        if (k == CTL_PAIRS - 1) {
            if (early && A.eos_token >= 0 && A.eos_token < V) E::store(row + A.eos_token, -INFINITY);
            continue;
        }
        const bool bad = k < SAMD_BAD_MAX_SEQS;
        if (!bad && !early) continue;
        const int kk = bad ? k : k - SAMD_BAD_MAX_SEQS;
        const int len = bad ? s_bad_len[kk] : s_stop_len[kk];
        if (len <= 0 || len > SAMD_BAD_MAX_LEN || len - 1 > n_ctx) continue;
        const int *seq = (bad ? s_bad : s_stop) + kk * SAMD_BAD_MAX_LEN;
        const int *ctx = s_ctx[j] + CTX - (len - 1);
        bool hit = true;
        for (int i = 0; i < len - 1 && hit; ++i) hit = ctx[i] == seq[i];
        const int t = seq[len - 1];
        if (hit && t >= 0 && t < V) E::store(row + t, -INFINITY);
    }
}

template <int kDtype>
void launch(const samd_logit_control_args &a, cudaStream_t stream) {
    logit_controls_kernel<kDtype><<<a.batch, CTL_THREADS, 0, stream>>>(a);
}

}  // namespace

extern "C" int samd_apply_logit_controls(const samd_logit_control_args *a, void *stream) {
    SAMD_REQUIRE(a && a->logits_dev && a->bias_ids_dev && a->bias_dev && a->bias_n_dev && a->bad_tokens_dev &&
                 a->bad_len_dev && a->min_tokens_dev, "samd_apply_logit_controls: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->vocab > 0 && a->n_slots > 0, "samd_apply_logit_controls: bad shape");
    SAMD_REQUIRE(a->n_nodes > 0 && a->n_nodes <= CTL_MAX_NODES, "samd_apply_logit_controls: n_nodes must be in [1, 256]");
    SAMD_REQUIRE(!a->retrieve_dev || (a->tokens_dev && a->n_paths > 0 && a->depth > 0),
                 "samd_apply_logit_controls: a path table needs the node tokens and a positive shape");
    SAMD_REQUIRE(!a->hist_len_dev || (a->hist_dev && a->hist_stride > 0),
                 "samd_apply_logit_controls: a history length needs the history");
    SAMD_REQUIRE(!a->stop_tokens_dev == !a->stop_len_dev, "samd_apply_logit_controls: stop tokens and lengths go together");
    SAMD_REQUIRE(a->dtype == SAMD_DTYPE_BF16 || a->dtype == SAMD_DTYPE_FP16 || a->dtype == SAMD_DTYPE_FP32,
                 "samd_apply_logit_controls: bad dtype");
    if (a->dtype == SAMD_DTYPE_BF16) launch<SAMD_DTYPE_BF16>(*a, (cudaStream_t)stream);
    else if (a->dtype == SAMD_DTYPE_FP16) launch<SAMD_DTYPE_FP16>(*a, (cudaStream_t)stream);
    else launch<SAMD_DTYPE_FP32>(*a, (cudaStream_t)stream);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
