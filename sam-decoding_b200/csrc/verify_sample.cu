// Stochastic (typical-acceptance) tree verification - the sampling branch of eval_posterior (samd/utils.py:142-184)
// together with the token draw that follows it (gen_candidates, samd/utils.py:85-88: torch.multinomial(sample_p, 1)).
//
// One CTA per request.  The reference walks the draft level by level: among the paths that share the accepted prefix,
// each distinct candidate token x of level i is tested once, in path order, with one uniform draw r against
//     p(x) / (1 - mass already rejected at this level),        p = softmax(logits_processor(logits[fi, i-1]))
// (logits_processor = temperature, then top-p, then top-k: SamdGenerationConfig.prepare_logits_processor, :44-58); the
// first accepted x extends the prefix, a rejected x is removed from the level's distribution.  The token after the
// accepted prefix is drawn from the level's residual distribution if its last level rejected something, otherwise from the
// plain softmax of the last accepted node's row (no processor - the reference's own asymmetry, :176-179).
//
// RNG contract (samd_b200.h): Philox4x32-10; uniform number k of request b is
//     u = (philox(counter = {lo32(off_b + k), hi32(off_b + k), 0, 0}, key = {lo32(seed_b), hi32(seed_b)})[0] >> 8) * 2^-24
// - one draw per tested candidate, then one for the next token; offsets_dev[b] is advanced by the number of draws used.
// The walk is replicated on every thread of the CTA (same data, same draws): the threads only cooperate on the passes
// over the vocabulary (maximum, the top-p / top-k thresholds by bisection over order-preserving keys, the normaliser, and
// the inverse-CDF draw).
//
// Per-request arguments (samd_verify_sample_requests): the processor (temperature, top-p, top-k) is read per request; a
// greedy request follows the greedy eval_posterior (samd/utils.py:127-141) and makes no draw; a finished request (done, or
// no live path) exits at once with accept_len 0 and no draw; a request's walk stops at its own path width and a -1 wraps
// to its own last row, so the pad columns of a table narrower than the batch's are never compared.
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <string.h>

#define ST 256                 // threads per CTA
#define MAX_REJ 64             // distinct rejected tokens of a level listed in shared memory (see kWide)
#define MAX_GREEDY_T 256       // node rows of a request with greedy requests in the launch

struct PhiloxState {
    uint32_t k0, k1;
    unsigned long long off;
    int used;
};

__device__ __forceinline__ float philox_uniform(PhiloxState &s) {
    const unsigned long long ctr = s.off + (unsigned long long)s.used++;
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = 0, c3 = 0;
    uint32_t k0 = s.k0, k1 = s.k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return (float)(c0 >> 8) * (1.0f / 16777216.0f);
}

__device__ __forceinline__ uint32_t skey(float f) {          // order-preserving key of a finite float (NaN -> max)
    const uint32_t b = __float_as_uint(f), a = b & 0x7FFFFFFFu;
    if (a > 0x7F800000u) return 0xFFFFFFFFu;
    if (a == 0) return 0x80000000u;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

template <int kDtype>
__device__ __forceinline__ float logit_at(const void *base, size_t i) {
    if (kDtype == SAMD_DTYPE_FP32) return __ldg(reinterpret_cast<const float *>(base) + i);
    if (kDtype == SAMD_DTYPE_BF16) return __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16 *>(base) + i));
    return __half2float(__ldg(reinterpret_cast<const __half *>(base) + i));
}

template <typename F>
__device__ __forceinline__ F block_sum(F v, F *s_red) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(SAMD_FULL, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    F t = 0;
    for (int w = 0; w < ST / 32; ++w) t += s_red[w];          // same order on every thread: identical result everywhere
    return t;
}
__device__ __forceinline__ float block_max(float v, float *s_red) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(SAMD_FULL, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = s_red[0];
    for (int w = 1; w < ST / 32; ++w) t = fmaxf(t, s_red[w]);
    return t;
}
__device__ __forceinline__ uint32_t block_min_u32(uint32_t v, int *s_scratch) {
    for (int o = 16; o; o >>= 1) v = min(v, (uint32_t)__shfl_xor_sync(SAMD_FULL, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_scratch[threadIdx.x >> 5] = (int)v;
    __syncthreads();
    uint32_t t = (uint32_t)s_scratch[0];
    for (int w = 1; w < ST / 32; ++w) t = min(t, (uint32_t)s_scratch[w]);
    __syncthreads();
    return t;
}
__device__ __forceinline__ float key_float(uint32_t k) {     // inverse of skey for the keys of finite values
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// a row's distribution: p(x) = kept(x) ? exp((l(x) - m) * inv_t) / z : 0.  kept(x): key(l(x)) >= thr, except the first
// tokens (index < pidx) of the tie group with key pkey, which top-p removed (pidx 0: none)
struct RowDist {
    float m, inv_t, z;
    uint32_t thr, pkey;
    int pidx;
};
__device__ __forceinline__ bool kept(const RowDist &d, uint32_t k, int i) {
    return k >= d.thr && !(k == d.pkey && i < d.pidx);
}

// Masses are sums of expf (not __expf) in double: where top-p cuts depends on them, and at V = 128256 one tail token
// holds ~1e-5 of the mass - float32 sums of 10^5 terms are off by that much.
template <int kDtype>
__device__ RowDist row_dist(const void *logits, size_t off, int V, bool processed, float temperature, float top_p, int top_k,
                            float *s_red, double *s_redd, int *s_cnt) {
    RowDist d;
    d.inv_t = processed ? 1.0f / temperature : 1.0f;
    d.thr = d.pkey = 0;
    d.pidx = 0;
    float m = -INFINITY;
    for (int i = threadIdx.x; i < V; i += ST) m = fmaxf(m, logit_at<kDtype>(logits, off + i));
    d.m = block_max(m, s_red);
    auto mass = [&](uint32_t lo_key, bool below) {            // sum of exp over key <= lo_key (below) or key >= lo_key
        double acc = 0.0;
        for (int i = threadIdx.x; i < V; i += ST) {
            const float l = logit_at<kDtype>(logits, off + i);
            const uint32_t k = skey(l);
            if (below ? k <= lo_key : k >= lo_key) acc += (double)expf((l - d.m) * d.inv_t);
        }
        return block_sum(acc, s_redd);
    };
    if (processed) {
        const uint32_t kmax = skey(d.m);
        uint32_t keep_from = 0;                               // keys >= keep_from survive
        int cut = 0;                                          // members of the tie group pkey that top-p removed
        if (top_p >= 1e-8f && top_p < 1.0f) {
            // TopPLogitsWarper: ascending cumulative probability <= 1 - top_p is removed (the maximum always stays):
            // the largest key K with mass(key <= K) <= (1 - top_p) * total, found by bisection over the key space
            const double total = mass(0u, false);
            const double budget = (1.0 - (double)top_p) * total;
            uint32_t lo = 0, hi = kmax - 1;                    // invariant: mass(<= lo) <= budget (lo = 0: below every key)
            while (lo < hi) {
                const uint32_t mid = lo + (uint32_t)(((unsigned long long)hi - lo + 1) >> 1);
                if (mass(mid, true) <= budget) lo = mid;
                else hi = mid - 1;
            }
            keep_from = lo + 1;
            // the tie group just above the cut: the ascending sort (stable: equal values in index order) removes its
            // first members while the cumulative mass stays within the budget - 16-bit logits tie in large groups
            uint32_t k2 = 0xFFFFFFFFu;
            for (int i = threadIdx.x; i < V; i += ST) {
                const uint32_t k = skey(logit_at<kDtype>(logits, off + i));
                if (k > lo && k < k2) k2 = k;
            }
            k2 = block_min_u32(k2, s_cnt);
            const double e = (double)expf((key_float(k2) - d.m) * d.inv_t);
            const double room = budget - mass(lo, true);
            const double fc = room > 0.0 ? floor(room / e) : 0.0;
            const int chunk = (V + ST - 1) / ST;              // members counted per contiguous chunk, in index order
            const int x0 = threadIdx.x * chunk, x1 = min(V, x0 + chunk);
            int n = 0;
            for (int x = x0; x < x1; ++x) n += skey(logit_at<kDtype>(logits, off + x)) == k2;
            s_cnt[threadIdx.x] = n;
            __syncthreads();
            int size = 0;
            for (int t = 0; t < ST; ++t) size += s_cnt[t];
            cut = (int)fmin(fc, (double)(size - 1));          // the maximum's last member always stays
            int before = 0, owner = -1;
            for (int t = 0; t < ST && cut > 0; ++t) {
                if (before + s_cnt[t] >= cut) {
                    owner = t;
                    break;
                }
                before += s_cnt[t];
            }
            __syncthreads();
            if (threadIdx.x == owner) {                       // index just past the cut-th member
                int seen = before, x = x0;
                for (; x < x1; ++x)
                    if (skey(logit_at<kDtype>(logits, off + x)) == k2 && ++seen == cut) break;
                s_cnt[0] = x + 1;
            }
            __syncthreads();
            if (cut > 0) {
                d.pkey = k2;
                d.pidx = s_cnt[0];
            }
            __syncthreads();
        }
        if (top_k > 0) {
            // TopKLogitsWarper on what is left: everything below the k-th largest surviving value goes (ties stay)
            auto count_ge = [&](uint32_t key) {
                float c = 0.f;
                for (int i = threadIdx.x; i < V; i += ST) c += skey(logit_at<kDtype>(logits, off + i)) >= key ? 1.f : 0.f;
                return block_sum(c, s_red) - (key <= d.pkey ? (float)cut : 0.f);
            };
            if (count_ge(keep_from) > (float)top_k) {
                uint32_t lo = keep_from, hi = kmax;            // largest key with count(>= key) >= k
                while (lo < hi) {
                    const uint32_t mid = lo + (uint32_t)(((unsigned long long)hi - lo + 1) >> 1);
                    if (count_ge(mid) >= (float)top_k) lo = mid;
                    else hi = mid - 1;
                }
                keep_from = lo;
            }
        }
        d.thr = keep_from;
    }
    double z = 0.0;
    for (int i = threadIdx.x; i < V; i += ST) {
        const float l = logit_at<kDtype>(logits, off + i);
        if (kept(d, skey(l), i)) z += (double)expf((l - d.m) * d.inv_t);
    }
    d.z = (float)block_sum(z, s_redd);
    return d;
}

template <int kDtype>
__device__ __forceinline__ float prob_of(const RowDist &d, const void *logits, size_t off, int x) {
    const float l = logit_at<kDtype>(logits, off + x);
    return kept(d, skey(l), x) ? expf((l - d.m) * d.inv_t) / d.z : 0.f;
}

// torch.argmax of one row (lowest index among equal maxima, NaN is the maximum, +0 == -0), every thread gets it
template <int kDtype>
__device__ int row_argmax(const void *logits, size_t off, int V, unsigned long long *s_red64) {
    unsigned long long best = 0;                                // (key << 32) | ~index: max = largest key, then lowest index
    for (int i = threadIdx.x; i < V; i += ST) {
        const unsigned long long k = ((unsigned long long)skey(logit_at<kDtype>(logits, off + i)) << 32) | (0xFFFFFFFFu - (uint32_t)i);
        best = k > best ? k : best;
    }
    for (int o = 16; o; o >>= 1) {
        const unsigned long long v = __shfl_xor_sync(SAMD_FULL, best, o);
        best = v > best ? v : best;
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red64[threadIdx.x >> 5] = best;
    __syncthreads();
    unsigned long long t = s_red64[0];
    for (int w = 1; w < ST / 32; ++w) t = s_red64[w] > t ? s_red64[w] : t;
    return (int)(0xFFFFFFFFu - (uint32_t)t);
}

struct SampleParams {
    samd_sample_args a;
    samd_sample_request_args r;                                 // every pointer NULL: the shared scalars of `a`
};

// Until a level accepts, every candidate tested there is rejected: at level `level`, token x has been rejected before
// path `upto` iff it is cand(p', level) of an earlier path p' that shares path prefix_of's first `level` tokens
// (candidate_tokens = tokens_ext[retrieve]: -1 picks the appended 0, as in the kernel's cand)
__device__ __forceinline__ bool level_has(const samd_sample_args &A, int b, const int32_t *tok, int x, int upto, int level,
                                          int prefix_of) {
    auto cand = [&](int p, int j) {
        const int r = A.retrieve_dev ? A.retrieve_dev[(size_t)b * A.retrieve_batch_stride + (size_t)p * A.depth + j] : j;
        return r < 0 ? 0 : tok[r];
    };
    for (int p = 0; p < upto; ++p) {
        if (cand(p, level) != x) continue;
        bool eq = true;
        for (int j = 0; j < level && eq; ++j) eq = cand(p, j) == cand(prefix_of, j);
        if (eq) return true;
    }
    return false;
}

// kWide: the path table has more than MAX_REJ paths, so a level may reject more tokens than s_rej lists.  Then a
// token past the list is found in the path table with level_has.  That costs up to n_paths prefix
// comparisons for every kept token in each of the three passes over the vocabulary - slow, but only a caller passing
// more than 64 paths through the C ABI gets there (the batched decoders' trees have at most 8 children per node), and
// the host picks this instantiation from the table's width, so the common one compiles without it.
template <int kDtype, bool kWide>
__global__ void __launch_bounds__(ST) verify_sample_kernel(SampleParams P) {
    __shared__ float s_red[ST / 32];
    __shared__ unsigned long long s_red64[ST / 32];
    __shared__ double s_redd[ST / 32];
    __shared__ int s_cnt[ST];
    __shared__ float s_part[ST];
    __shared__ int s_rej[MAX_REJ];
    __shared__ int s_am[MAX_GREEDY_T];
    const samd_sample_args &A = P.a;
    const samd_sample_request_args &R = P.r;
    const int b = blockIdx.x;
    const int V = A.vocab;
    const int T = R.n_nodes_dev ? R.n_nodes_dev[b] : A.n_nodes;           // this request's rows: -1 wraps to row T - 1
    const int n_paths = A.retrieve_dev ? (A.n_paths_dev ? A.n_paths_dev[b] : A.n_paths) : 1;
    const int width = A.retrieve_dev ? A.depth : A.n_nodes;                 // the table's width = the output stride
    const int depth = max(1, min(width, R.depth_dev ? R.depth_dev[b] : A.retrieve_dev ? A.depth : T));
    if ((R.done_dev && R.done_dev[b]) || n_paths <= 0) {                    // finished: no draw, nothing but accept_len 0
        if (threadIdx.x == 0 && A.out_accept_len_dev) A.out_accept_len_dev[b] = 0;
        return;
    }
    const int32_t *tok = A.tree_tokens_dev + (size_t)b * A.n_nodes;
    auto ri = [&](int p, int j) { return A.retrieve_dev ? A.retrieve_dev[(size_t)b * A.retrieve_batch_stride + (size_t)p * A.depth + j] : j; };
    auto cand = [&](int p, int j) {                             // candidate_tokens = tokens_ext[retrieve]: -1 picks the appended 0
        const int r = ri(p, j);
        return r < 0 ? 0 : tok[r];
    };
    auto row_off = [&](int p, int j) {                          // logits[retrieve]: -1 wraps to the request's last row
        const int r = ri(p, j);
        return (size_t)b * A.batch_stride + (size_t)(r < 0 ? T - 1 : r) * A.row_stride;
    };
    auto emit_path = [&](int best, int accept_len) {            // accepted tokens and indices, -1 past accept_len
        for (int j = threadIdx.x; j < width; j += ST) {
            if (A.out_tokens_dev) A.out_tokens_dev[(size_t)b * width + j] = j < accept_len ? cand(best, j) : -1;
            if (A.out_indices_dev) A.out_indices_dev[(size_t)b * width + j] = j < accept_len ? ri(best, j) : -1;
        }
    };
    if (R.greedy_dev && R.greedy_dev[b]) {
        // greedy eval_posterior: the argmax of every row, each path's match length, the first longest path, and the
        // argmax of its last accepted row as the next token
        for (int t = 0; t < T; ++t) {
            const int am = row_argmax<kDtype>(A.logits_dev, (size_t)b * A.batch_stride + (size_t)t * A.row_stride, V, s_red64);
            if (threadIdx.x == 0) s_am[t] = am;
        }
        __syncthreads();
        int best = 0, acc = 0;
        for (int p = 0; p < n_paths; ++p) {
            int a = 0;
            for (int j = 0; j + 1 < depth; ++j) {
                const int r = ri(p, j);
                if (cand(p, j + 1) != s_am[r < 0 ? T - 1 : r]) break;
                ++a;
            }
            if (a > acc) acc = a, best = p;
        }
        if (threadIdx.x == 0) {
            const int r = ri(best, acc);
            if (A.out_best_dev) A.out_best_dev[b] = best;
            if (A.out_accept_len_dev) A.out_accept_len_dev[b] = acc + 1;
            if (A.out_next_token_dev) A.out_next_token_dev[b] = s_am[r < 0 ? T - 1 : r];
        }
        emit_path(best, acc + 1);
        return;
    }
    const float temperature = R.temperature_dev ? R.temperature_dev[b] : A.temperature;
    const float top_p = R.top_p_dev ? R.top_p_dev[b] : A.top_p;
    const int top_k = R.top_k_dev ? R.top_k_dev[b] : A.top_k;
    PhiloxState rng;
    {
        const unsigned long long seed = A.seeds_dev[b];
        rng.k0 = (uint32_t)seed;
        rng.k1 = (uint32_t)(seed >> 32);
        rng.off = A.offsets_dev[b];
        rng.used = 0;
    }
    int accept_len = 1, best = 0, n_rej = 0;                    // n_rej: rejected tokens of the level (kWide: all)
    bool adjust = false;
    RowDist dist;                                               // the last level's processed distribution
    size_t dist_off = 0;
    for (int i = 1; i < depth; ++i) {
        if (i != accept_len) break;
        adjust = false;
        n_rej = 0;
        // the paths that share the accepted prefix (the prefix is path `best`'s); the first of them supplies the row
        int fi = -1;
        for (int p = 0; p < n_paths && fi < 0; ++p) {
            bool eq = true;
            for (int j = 0; j < accept_len && eq; ++j) eq = cand(p, j) == cand(best, j);
            if (eq) fi = p;
        }
        dist_off = row_off(fi, i - 1);
        dist = row_dist<kDtype>(A.logits_dev, dist_off, V, true, temperature, top_p, top_k, s_red, s_redd, s_cnt);
        float rej_mass = 0.f;
        const int prefix_of = best;
        for (int p = 0; p < n_paths; ++p) {
            bool eq = true;
            for (int j = 0; j < accept_len && eq; ++j) eq = cand(p, j) == cand(prefix_of, j);
            if (!eq) continue;
            const int x = cand(p, i);
            bool seen = false;
            if constexpr (kWide) {
                for (int q = 0; q < min(n_rej, MAX_REJ); ++q) seen |= s_rej[q] == x;
                if (!seen && n_rej > MAX_REJ) seen = level_has(A, b, tok, x, p, i, best);
            } else {
                for (int q = 0; q < n_rej; ++q) seen |= s_rej[q] == x;
            }
            if (seen) continue;
            const float r = philox_uniform(rng);
            const float px = prob_of<kDtype>(dist, A.logits_dev, dist_off, x) / (1.0f - rej_mass);
            if (r <= px) {
                accept_len += 1;
                best = p;
                break;
            }
            rej_mass += prob_of<kDtype>(dist, A.logits_dev, dist_off, x);
            __syncthreads();
            if (threadIdx.x == 0 && n_rej < MAX_REJ) s_rej[n_rej] = x;
            __syncthreads();
            if constexpr (kWide) n_rej += 1;
            else n_rej = min(n_rej + 1, MAX_REJ);
            adjust = true;
        }
    }
    // the distribution of the next token (samd/utils.py:173-179)
    const bool residual = adjust && accept_len != depth;
    if (!residual) {
        dist_off = row_off(best, accept_len - 1);
        dist = row_dist<kDtype>(A.logits_dev, dist_off, V, false, 1.0f, 0.f, 0, s_red, s_redd, s_cnt);
        n_rej = 0;
    }
    auto p_next = [&](int x) {
        if constexpr (kWide) {
            for (int q = 0; q < min(n_rej, MAX_REJ); ++q)
                if (s_rej[q] == x) return 0.f;
            const float px = prob_of<kDtype>(dist, A.logits_dev, dist_off, x);
            return n_rej > MAX_REJ && px > 0.f && level_has(A, b, tok, x, n_paths, accept_len, best) ? 0.f : px;
        } else {
            for (int q = 0; q < n_rej; ++q)
                if (s_rej[q] == x) return 0.f;
            return prob_of<kDtype>(dist, A.logits_dev, dist_off, x);
        }
    };
    // inverse-CDF draw in index order: contiguous blocks per thread, a scan over the blocks, then inside the block
    const int chunk = (V + ST - 1) / ST;
    const int x0 = threadIdx.x * chunk, x1 = min(V, x0 + chunk);
    float local = 0.f;
    for (int x = x0; x < x1; ++x) local += p_next(x);
    s_part[threadIdx.x] = local;
    __syncthreads();
    float total = 0.f;
    for (int t = 0; t < ST; ++t) total += s_part[t];
    const float u = philox_uniform(rng) * total;
    float before = 0.f;
    int owner = ST - 1;
    for (int t = 0; t < ST; ++t) {
        if (u < before + s_part[t]) {
            owner = t;
            break;
        }
        before += s_part[t];
    }
    if (A.out_sample_p_dev)
        for (int x = x0; x < x1; ++x) A.out_sample_p_dev[(size_t)b * V + x] = p_next(x) / total;
    if (threadIdx.x == owner) {
        float c = before;
        int pick = -1, last_pos = -1;
        for (int x = x0; x < x1; ++x) {
            const float px = p_next(x);
            if (px > 0.f) last_pos = x;
            c += px;
            if (u < c && px > 0.f) {
                pick = x;
                break;
            }
        }
        if (pick < 0) pick = last_pos >= 0 ? last_pos : max(0, x1 - 1);     // rounding at the very end of the block
        if (A.out_next_token_dev) A.out_next_token_dev[b] = pick;
    }
    if (threadIdx.x == 0) {
        if (A.out_best_dev) A.out_best_dev[b] = best;
        if (A.out_accept_len_dev) A.out_accept_len_dev[b] = accept_len;
        A.offsets_dev[b] = rng.off + (unsigned long long)rng.used;
    }
    emit_path(best, accept_len);
}

extern "C" int samd_verify_sample_requests(const samd_sample_args *a, const samd_sample_request_args *r, void *stream) {
    SAMD_REQUIRE(a && a->logits_dev && a->tree_tokens_dev && a->seeds_dev && a->offsets_dev, "samd_verify_sample: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->n_nodes > 0 && a->vocab > 0, "samd_verify_sample: bad shape");
    SAMD_REQUIRE(a->temperature >= 1e-5f, "samd_verify_sample: temperature must be >= 1e-5 (samd/utils.py:41)");
    SAMD_REQUIRE(!a->retrieve_dev || (a->n_paths > 0 && a->depth > 0), "samd_verify_sample: bad retrieve table shape");
    SAMD_REQUIRE(a->dtype == SAMD_DTYPE_BF16 || a->dtype == SAMD_DTYPE_FP16 || a->dtype == SAMD_DTYPE_FP32, "samd_verify_sample: bad dtype");
    SAMD_REQUIRE(!r || !r->greedy_dev || a->n_nodes <= MAX_GREEDY_T, "samd_verify_sample_requests: greedy requests need n_nodes <= 256");
    SampleParams P;
    P.a = *a;
    if (r) P.r = *r;
    else memset(&P.r, 0, sizeof(P.r));
    // a level can reject more than MAX_REJ distinct tokens only if the table has more paths than that
    const bool wide = a->retrieve_dev && a->n_paths > MAX_REJ;
    auto kern = a->dtype == SAMD_DTYPE_BF16 ? (wide ? verify_sample_kernel<SAMD_DTYPE_BF16, true> : verify_sample_kernel<SAMD_DTYPE_BF16, false>)
                : a->dtype == SAMD_DTYPE_FP16 ? (wide ? verify_sample_kernel<SAMD_DTYPE_FP16, true> : verify_sample_kernel<SAMD_DTYPE_FP16, false>)
                : (wide ? verify_sample_kernel<SAMD_DTYPE_FP32, true> : verify_sample_kernel<SAMD_DTYPE_FP32, false>);
    kern<<<a->batch, ST, 0, (cudaStream_t)stream>>>(P);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int samd_verify_sample(const samd_sample_args *a, void *stream) { return samd_verify_sample_requests(a, nullptr, stream); }
