// Fused greedy tree verification + KV-cache compaction, one persistent launch (sm_100a).
//
// Work is warp-granular over a grid that is fully resident (two grid-wide barriers):
//   phase 1   item = a chunk (about 16k elements) of one logits row, handed out dynamically from 64 work queues.
//             A warp streams its chunk with 128-bit no-allocate loads (8 in flight per lane), keeps a WARP-uniform
//             running (key, index) maximum under torch.argmax's rule (lowest index among equal maxima, NaN is the
//             maximum, +0 == -0) - no block barrier, no shared memory - and publishes it with a fire-and-forget
//             64-bit atomicMax.  Nothing in the loop waits on a round trip but the logits themselves.
//   barrier A every row maximum is published.
//   phase 1b  one warp per request walks the P x D path table (samd/utils.py:127-141), writes best / accept_len /
//             next_token / accepted tokens + indices, snapshots and bumps cache_len and, if rows have to move,
//             appends a move record to the active list.
//   barrier B every walk is published.
//   phase 2   the moved rows of the active requests are flattened into 16-byte units over every lane of the grid:
//             rows cache_len+indices[j] -> cache_len+j (samd/cache.py:118-133) for all heads, loads of a row group
//             before its stores (the reference gathers into a temporary first; ascending j with indices[j] >= j
//             makes that order equivalent).
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>

#define VT 256                 // threads per CTA (8 warps)
#define VW (VT / 32)
#define UNROLL 8               // 128-bit loads in flight per lane
#define KV_GROUP 8             // accepted rows staged in registers per pass
#define KV_REC (3 + KV_GROUP)   // move record: {request, accept_len, start, first KV_GROUP source rows}

struct samd_verify_s {
    unsigned long long *node_key;   // [max_batch][max_nodes]
    int *active;                    // [max_batch][KV_REC] move records of the requests with rows to move
    int *counters;                  // [CN_WORDS] epoch, exit count, work counter, barrier arrivals and flags, n_active
    int occ_per_sm[6];              // cached occupancy per dtype (x top-k variant)
    unsigned long long *topk_part;  // [topk_items][TOPK] per-chunk top-8 lists
    long long topk_items;
    int *kv_start;                  // [max_batch] cache_len before the bump
    int *req_done, *act_flag;       // [max_batch] each (overlapped flow)
    int max_batch, max_nodes, device, n_sms;
};

struct VerifyParams {
    samd_verify_args a;
    unsigned long long *node_key;
    int *active, *counters, *kv_start;
    int *req_done;                   // [max_batch] items of the request that have reported (overlapped flow)
    int *act_flag;                   // [max_batch] launch epoch once move record [slot] is complete (overlapped flow)
    int overlap;                     // 1 = walks as requests complete, ticketed row moves, no grid barrier
    int max_nodes, max_batch;
    int chunk, chunks_per_row, n_items1, n_items2, vec_ok, stage_cap;
    int p1_warps;                    // warps that take part in phase 1 (<= the grid's warps)
    int tma;                         // 1 = phase 1 stages the logits through shared memory with the bulk-copy engine
    int ring_off;                    // byte offset of the staging rings in dynamic shared memory (128-byte aligned)
    unsigned long long *topk_part;   // [n_items1][TOPK] per-chunk lists (top-k launches)
    unsigned long long *dbg_times;   // optional [grid warps][3] globaltimer ns: start, end of streaming, exit (profiling hook)
};

__device__ __forceinline__ unsigned long long samd_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

template <int kDtype>
__device__ __forceinline__ uint32_t orderable16(uint32_t b) {
    const uint32_t nan_above = kDtype == SAMD_DTYPE_BF16 ? 0x7F80u : 0x7C00u;
    const uint32_t a = b & 0x7FFFu;
    if (a > nan_above) return 0xFFFFu;            // any NaN is the maximum
    if (a == 0) return 0x8000u;                   // +0 == -0
    return (b & 0x8000u) ? (~b & 0xFFFFu) : (b | 0x8000u);
}

template <int kDtype>
__device__ __forceinline__ uint32_t vec_max_bits(const uint4 &x) {
    if (kDtype == SAMD_DTYPE_BF16) {
        __nv_bfloat162 a = __hmax2_nan(*reinterpret_cast<const __nv_bfloat162 *>(&x.x),
                                       *reinterpret_cast<const __nv_bfloat162 *>(&x.y));
        __nv_bfloat162 b = __hmax2_nan(*reinterpret_cast<const __nv_bfloat162 *>(&x.z),
                                       *reinterpret_cast<const __nv_bfloat162 *>(&x.w));
        a = __hmax2_nan(a, b);
        __nv_bfloat16 s = __hmax_nan(__low2bfloat16(a), __high2bfloat16(a));
        return (uint32_t)__bfloat16_as_ushort(s);
    } else {
        __half2 a = __hmax2_nan(*reinterpret_cast<const __half2 *>(&x.x), *reinterpret_cast<const __half2 *>(&x.y));
        __half2 b = __hmax2_nan(*reinterpret_cast<const __half2 *>(&x.z), *reinterpret_cast<const __half2 *>(&x.w));
        a = __hmax2_nan(a, b);
        __half s = __hmax_nan(__low2half(a), __high2half(a));
        return (uint32_t)__half_as_ushort(s);
    }
}

__device__ __forceinline__ uint32_t orderable32(uint32_t b) {
    const uint32_t a = b & 0x7FFFFFFFu;
    if (a > 0x7F800000u) return 0xFFFFFFFFu;      // NaN is the maximum
    if (a == 0) return 0x80000000u;               // +0 == -0
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// NaN-propagating packed maximum of two 16-bit pairs held as raw bits (HMNMX2 on sm_100a)
template <int kDtype>
__device__ __forceinline__ uint32_t hmax2_bits(uint32_t a, uint32_t b) {
    if (kDtype == SAMD_DTYPE_BF16) {
        const __nv_bfloat162 r = __hmax2_nan(*reinterpret_cast<const __nv_bfloat162 *>(&a), *reinterpret_cast<const __nv_bfloat162 *>(&b));
        return *reinterpret_cast<const uint32_t *>(&r);
    } else {
        const __half2 r = __hmax2_nan(*reinterpret_cast<const __half2 *>(&a), *reinterpret_cast<const __half2 *>(&b));
        return *reinterpret_cast<const uint32_t *>(&r);
    }
}

template <int kDtype>
__device__ __forceinline__ uint32_t vec_pair_max(const uint4 &x) {
    return hmax2_bits<kDtype>(hmax2_bits<kDtype>(x.x, x.y), hmax2_bits<kDtype>(x.z, x.w));
}

// orderable key of the larger half of a packed pair
template <int kDtype>
__device__ __forceinline__ uint32_t pair_key(uint32_t m) {
    const uint32_t a = orderable16<kDtype>(m & 0xFFFFu), b = orderable16<kDtype>(m >> 16);
    return a > b ? a : b;
}

__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

template <int kDtype>
__device__ __forceinline__ void fold_vec(const uint4 &x, uint32_t elem, uint32_t &best_key, uint32_t &best_idx) {
    const uint32_t k = orderable16<kDtype>(vec_max_bits<kDtype>(x));
    if (k > best_key) {                            // rare after the first few vectors
        const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const uint32_t ke = orderable16<kDtype>((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu);
            if (ke > best_key) {
                best_key = ke;
                best_idx = elem + e;
            }
        }
    }
}

// ---- bulk-copy engine (TMA) staging: global -> shared with an mbarrier per stage ---------------------------------
#define TMA_STAGES 4           // groups (2 KB each) in flight per warp
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

template <int G>
__device__ __forceinline__ void load_group(uint4 (&x)[G], const uint4 *v4, int v0, int nvec, int lane, uint32_t ninf) {
#pragma unroll
    for (int u = 0; u < G; ++u) {
        const int vi = v0 + u * 32 + lane;
        x[u] = vi < nvec ? ld_stream(v4 + vi) : make_uint4(ninf, ninf, ninf, ninf);
    }
}

// Fold one group of 32 x G vectors into the WARP-uniform running maximum (best_key, best_idx).
template <int kDtype, int G>
__device__ __forceinline__ void fold_group(const uint4 (&x)[G], int v0, int nvec, int lane, int e0, uint32_t &best_key,
                                           uint32_t &best_idx) {
    uint32_t m = vec_pair_max<kDtype>(x[0]);
#pragma unroll
    for (int u = 1; u < G; ++u) m = hmax2_bits<kDtype>(m, vec_pair_max<kDtype>(x[u]));
    const uint32_t wk = __reduce_max_sync(SAMD_FULL, pair_key<kDtype>(m));
    if (wk <= best_key) return;                                // warp-uniform; taken ~ln(#groups) times per row
    best_key = wk;
    bool found = false;
#pragma unroll
    for (int u = 0; u < G; ++u) {
        if (found) continue;
        const int vi = v0 + u * 32 + lane;
        const unsigned bal = __ballot_sync(SAMD_FULL, vi < nvec && pair_key<kDtype>(vec_pair_max<kDtype>(x[u])) == wk);
        if (bal) {                                             // lowest u, then lowest lane = lowest index
            found = true;
            const int src = __ffs(bal) - 1;
            int e_first = 0;
            if (lane == src) {
                const uint32_t w[4] = {x[u].x, x[u].y, x[u].z, x[u].w};
                e_first = 7;
#pragma unroll
                for (int e = 7; e >= 0; --e)
                    if (orderable16<kDtype>((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu) == wk) e_first = e;
            }
            e_first = __shfl_sync(SAMD_FULL, e_first, src);
            best_idx = (uint32_t)(e0 + (v0 + u * 32 + src) * 8 + e_first);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Top-8 per row (Token Recycle, samd/tree_model/token_recycle/token_recycle.py:36-38) in the same pass.
// The warp keeps a sorted list of 8 composites  key << 32 | (0xFFFFFFFF - index)  in lanes 0..7 (descending:
// value descending, index ascending - lane 0 is the argmax) and the warp-uniform key of the 8th entry as the
// admission threshold; elements equal to -inf never enter (a row with fewer than 8 larger elements is completed
// from a re-scan when the chunks are merged).
// ---------------------------------------------------------------------------------------
#define TOPK 8

template <int kDtype>
__device__ __forceinline__ uint32_t key_ninf() {
    return kDtype == SAMD_DTYPE_BF16 ? 0x007Fu : kDtype == SAMD_DTYPE_FP16 ? 0x03FFu : 0x007FFFFFu;
}

__device__ __forceinline__ void topk_insert(unsigned long long c, unsigned long long &t, uint32_t &thrv, int lane) {
    const int pos = __popc(__ballot_sync(SAMD_FULL, lane < TOPK && t > c));      // a prefix: the list is sorted
    const unsigned long long prev = __shfl_up_sync(SAMD_FULL, t, 1);
    if (lane < TOPK && lane >= pos) t = lane == pos ? c : prev;
    thrv = (uint32_t)(__shfl_sync(SAMD_FULL, t, TOPK - 1) >> 32);
}

// raw bits of a value v such that {x > v} contains {key(x) > T} (and nothing that could displace a list entry)
template <int kDtype>
__device__ __forceinline__ uint32_t threshold_bits(uint32_t T) {
    if (T == 0x7FFFu) return 0x8001u;                           // between the negatives and zero: just below -0
    return (T & 0x8000u) ? (T ^ 0x8000u) : (~T & 0xFFFFu);
}

// per-half "x > v or unordered" mask of one packed word (0xFFFF per true half)
template <int kDtype>
__device__ __forceinline__ uint32_t gtu_mask(uint32_t w, uint32_t v2) {
    if (kDtype == SAMD_DTYPE_BF16)
        return __hgtu2_mask(*reinterpret_cast<const __nv_bfloat162 *>(&w), *reinterpret_cast<const __nv_bfloat162 *>(&v2));
    return __hgtu2_mask(*reinterpret_cast<const __half2 *>(&w), *reinterpret_cast<const __half2 *>(&v2));
}

// Vector path.  Most groups are rejected by their packed maximum.  In a group that passes, every lane marks its
// elements above the threshold with packed compares (bit w = low half of its word w, bit 16 + w = high half; the
// lane's G vectors are words 0 .. 4G-1), then the marked elements are inserted - in any order: the list keeps the
// 8 largest composites of whatever it is fed.
template <int kDtype, int G>
__device__ __forceinline__ void fold_group_topk(const uint4 (&x)[G], int v0, int nvec, int lane, int e0, unsigned long long &t,
                                                uint32_t &thrv, uint32_t floorv) {
    static_assert(G == 4, "candidate masks hold 16 words per lane");
    uint32_t m = vec_pair_max<kDtype>(x[0]);
#pragma unroll
    for (int u = 1; u < G; ++u) m = hmax2_bits<kDtype>(m, vec_pair_max<kDtype>(x[u]));
    const uint32_t wk = __reduce_max_sync(SAMD_FULL, pair_key<kDtype>(m));
    const uint32_t T = max(thrv, floorv);
    if (wk <= T) return;                                        // warp-uniform
    const uint32_t v = threshold_bits<kDtype>(T), v2 = v | (v << 16);
    uint32_t cand = 0;
#pragma unroll
    for (int u = 0; u < G; ++u) {
        const uint32_t w[4] = {x[u].x, x[u].y, x[u].z, x[u].w};
        const bool live = v0 + u * 32 + lane < nvec;           // (padding lanes hold -inf and never pass anyway)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (live) cand |= (gtu_mask<kDtype>(w[i], v2) & 0x00010001u) << (u * 4 + i);
    }
    while (__any_sync(SAMD_FULL, cand != 0)) {
        // every lane with marks pops its lowest one and forms its composite
        unsigned long long c = 0;
        if (cand) {
            const int p = __ffs(cand) - 1, wsel = p & 15;
            cand &= cand - 1;
            uint32_t word = 0;
#pragma unroll
            for (int u = 0; u < G; ++u) {
                const uint32_t w[4] = {x[u].x, x[u].y, x[u].z, x[u].w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (wsel == u * 4 + i) word = w[i];
            }
            const uint32_t key = orderable16<kDtype>((p & 16) ? word >> 16 : word & 0xFFFFu);
            const uint32_t idx = (uint32_t)(e0 + (v0 + (wsel >> 2) * 32 + lane) * 8 + (wsel & 3) * 2 + (p >> 4));
            c = ((unsigned long long)key << 32) | (0xFFFFFFFFu - idx);
        }
        unsigned todo = __ballot_sync(SAMD_FULL, c != 0);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const unsigned long long cs = __shfl_sync(SAMD_FULL, c, src);
            if (cs > __shfl_sync(SAMD_FULL, t, TOPK - 1)) topk_insert(cs, t, thrv, lane);
        }
    }
}

// A lower bound for the admission threshold before the list has filled up: the group's 32 per-lane maxima are 32
// distinct elements, so nothing below the 8th largest of them can be among the chunk's top 8.  (Without it the
// first group alone feeds ~45 of a chunk's ~70 insertions.)  Returns a key k such that only keys > k can qualify.
template <int kDtype, int G>
__device__ __forceinline__ uint32_t topk_floor(const uint4 (&x)[G], int lane) {
    uint32_t m = vec_pair_max<kDtype>(x[0]);
#pragma unroll
    for (int u = 1; u < G; ++u) m = hmax2_bits<kDtype>(m, vec_pair_max<kDtype>(x[u]));
    const uint32_t mine = pair_key<kDtype>(m);
    int rank = 0;                                               // lanes with a larger maximum (ties: lower lane first)
#pragma unroll
    for (int l = 0; l < 32; ++l) {
        const uint32_t o = __shfl_sync(SAMD_FULL, mine, l);
        rank += (o > mine) || (o == mine && l < lane);
    }
    const unsigned who = __ballot_sync(SAMD_FULL, rank == TOPK - 1);
    const uint32_t eighth = __shfl_sync(SAMD_FULL, mine, __ffs(who) - 1);
    return max(key_ninf<kDtype>(), eighth - 1);                 // equal values may still qualify: strictly below
}

// Element-wise path (fp32, unaligned rows, ragged row ends): 32 consecutive elements, one per lane.
template <int kDtype>
__device__ __forceinline__ void fold_elems_topk(uint32_t ke, uint32_t idx, unsigned long long &t, uint32_t &thrv, int lane) {
    unsigned todo = __ballot_sync(SAMD_FULL, ke > max(thrv, key_ninf<kDtype>()));
    while (todo) {                                              // ascending lane = ascending index
        const int src = __ffs(todo) - 1;
        const uint32_t k = __shfl_sync(SAMD_FULL, ke, src), i = __shfl_sync(SAMD_FULL, idx, src);
        topk_insert(((unsigned long long)k << 32) | (0xFFFFFFFFu - i), t, thrv, lane);
        todo &= todo - 1;
        todo &= __ballot_sync(SAMD_FULL, ke > thrv);
    }
}

__device__ __forceinline__ int ri_at(const VerifyParams &P, int b, int p, int j) {
    if (!P.a.retrieve_dev) return j;                          // sequence: identity path
    return P.a.retrieve_dev[(size_t)b * P.a.retrieve_batch_stride + (size_t)p * P.a.depth + j];
}

// one unit of phase-1 work: a chunk of one logits row
struct Item {
    int item, b, t, e0, len;
    bool act;                                                  // rows past the request's node count stream nothing
};

__device__ __forceinline__ Item decode_item(const VerifyParams &P, int item) {
    Item I;
    I.item = item;
    I.act = false;
    I.b = I.t = I.e0 = I.len = 0;
    if (item >= P.n_items1) return I;
    const int C = P.chunks_per_row, T = P.a.n_nodes;
    const int row = item / C;
    I.e0 = (item - row * C) * P.chunk;
    I.len = min(P.chunk, P.a.vocab - I.e0);
    I.b = row / T;
    I.t = row - I.b * T;
    I.act = I.t < (P.a.n_nodes_dev ? P.a.n_nodes_dev[I.b] : T);
    return I;
}

__device__ __forceinline__ size_t item_offset(const VerifyParams &P, const Item &I) {
    return (size_t)I.b * P.a.batch_stride + (size_t)I.t * P.a.row_stride + I.e0;
}

// counters[] slots (all re-armed by the kernel itself, so a launch can be captured in a CUDA graph and replayed)
enum { CN_EPOCH = 0, CN_EXIT, CN_ARRIVE_A, CN_FLAG_A, CN_ARRIVE_B, CN_FLAG_B, CN_ACTIVE, CN_ARRIVE_C, CN_FLAG_C, CN_TICKET, CN_WALKS,
       CN_QUEUES = 32 };
// Work queues: one counter would be hit by every warp for every item, and same-address atomics serialise at about
// 3 ns each on B200 (measured: 62k items took 135 us whatever their size) - so the dynamic items are dealt round-robin
// into N_QUEUES queues, each with its own counter on its own 128-byte line.
#define N_QUEUES 64
#define QUEUE_STRIDE 32
#define CN_WORDS (CN_QUEUES + N_QUEUES * QUEUE_STRIDE)

template <int kDtype, bool kTopK>
__global__ void __launch_bounds__(VT, 4) verify_compact_kernel(VerifyParams P) {
    extern __shared__ int s_am_all[];                          // [VW][2][n_nodes] node argmax + tree tokens, one slab per warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_ctas = (int)gridDim.x;
    const int gwarp = warp * n_ctas + blockIdx.x;             // warp-major: consecutive items land on different SMs
    const int n_warps = n_ctas * VW;
    // The launch epoch lives in device memory (bumped by the last CTA to leave): nothing launch-specific is baked
    // into the kernel arguments.  Flags are written once per launch with the epoch value and only ever compared.
    const int epoch = *reinterpret_cast<volatile int *>(&P.counters[CN_EPOCH]) + 1;
    const samd_verify_args &A = P.a;
    const int T = A.n_nodes;
    const int C = P.chunks_per_row;
    unsigned long long *dbg = P.dbg_times ? P.dbg_times + ((size_t)blockIdx.x * VW + warp) * 3 : nullptr;
    if (dbg && lane == 0) dbg[0] = samd_globaltimer();
    int *s_am = s_am_all + warp * 2 * T;                     // [T] node argmax, then [T] tree tokens
    int *s_tok = s_am + T;
    const uint16_t *logits = reinterpret_cast<const uint16_t *>(A.logits_dev);

    // The walk of one request (samd/utils.py:127-141 + update_state + the move record), by one warp.
    auto walk_request = [&](int b) {
        // keys, tree tokens and this lane's path row are fetched together (one memory round trip); the walk
        // itself then runs out of shared memory and registers
        const int n_rows = A.n_nodes_dev ? A.n_nodes_dev[b] : T;
        const int32_t *tok = A.tree_tokens_dev + (size_t)b * T;
        const int n_paths = A.retrieve_dev ? (A.n_paths_dev ? A.n_paths_dev[b] : A.n_paths) : 1;
        const int depth = A.retrieve_dev ? A.depth : n_rows;
        constexpr int WD = 8;                                   // path depth held in registers
        // (a request with no live path - a finished one, samd_draft_assemble - takes the general walk: acc = 0, index 0 -> 0)
        const bool fast = A.retrieve_dev && depth <= WD && n_paths > 0 && n_paths <= 32;
        int rp[WD];
#pragma unroll
        for (int j = 0; j < WD; ++j) rp[j] = (fast && lane < n_paths && j < depth) ? ri_at(P, b, lane, j) : -1;
        int start = 0;
        if (lane == 0 && A.cache_len_dev) start = A.cache_len_dev[b];
        for (int i = lane; i < T; i += 32) {
            unsigned long long *kp = &P.node_key[(size_t)b * P.max_nodes + i];
            const unsigned long long k = __ldcg(kp);
            s_tok[i] = i < n_rows ? tok[i] : 0;
            const int am = (int)(0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull));
            s_am[i] = am;
            *kp = 0;                                            // re-arm for the next launch
            if (A.out_node_argmax_dev && i < n_rows) A.out_node_argmax_dev[(size_t)b * T + i] = am;
        }
        __syncwarp();
        unsigned int bestpk = 0;
        if (fast) {
            if (lane < n_paths) {
                int acc = 0;
#pragma unroll
                for (int j = 0; j + 1 < WD; ++j) {
                    if (j + 1 < depth && acc == j) {
                        const int rowi = rp[j] < 0 ? n_rows - 1 : rp[j];          // -1 wraps to the last row
                        const int cand = rp[j + 1] < 0 ? 0 : s_tok[rp[j + 1]];    // -1 selects the appended 0
                        if (cand == s_am[rowi]) acc++;
                    }
                }
                bestpk = ((unsigned)acc << 16) | (unsigned)(0xFFFF - lane);
            }
        } else {
            for (int p = lane; p < n_paths; p += 32) {
                int acc = 0;
                int prev = ri_at(P, b, p, 0);
                for (int j = 0; j + 1 < depth; ++j) {
                    const int nxt = ri_at(P, b, p, j + 1);
                    const int rowi = prev < 0 ? n_rows - 1 : prev;
                    const int cand = nxt < 0 ? 0 : s_tok[nxt];
                    if (cand != s_am[rowi]) break;
                    acc++;
                    prev = nxt;
                }
                bestpk = max(bestpk, ((unsigned)acc << 16) | (unsigned)(0xFFFF - p));   // max accept, first path
            }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) bestpk = max(bestpk, __shfl_xor_sync(SAMD_FULL, bestpk, o));
        const int acc = (int)(bestpk >> 16);
        const int best = acc == 0 ? 0 : (int)(0xFFFF - (bestpk & 0xFFFF));
        const int out_stride = A.retrieve_dev ? A.depth : T;
        int moved = 0, last = 0, ix0 = -1;                     // ix0: this lane's accepted index for j = lane
        for (int j0 = 0; j0 < out_stride; j0 += 32) {
            const int j = j0 + lane;
            int tk = -1, ix = -1;
            if (fast) {                                         // the best path's row is in that lane's registers
#pragma unroll
                for (int q = 0; q < WD; ++q) {
                    const int v = __shfl_sync(SAMD_FULL, rp[q], best);
                    if (lane == q) ix = v;
                }
                if (j > acc) ix = -1;
            } else if (j < out_stride && j <= acc) {
                ix = ri_at(P, b, best, j);
            }
            if (j < out_stride && j <= acc) {
                tk = ix < 0 ? 0 : s_tok[ix];
                moved += ix != j;
            }
            if (j < out_stride) {
                if (A.out_tokens_dev) A.out_tokens_dev[(size_t)b * out_stride + j] = tk;
                if (A.out_indices_dev) A.out_indices_dev[(size_t)b * out_stride + j] = ix;
            }
            if (j0 == 0) ix0 = ix;
            if (acc >= j0 && acc < j0 + 32) last = __shfl_sync(SAMD_FULL, ix, acc - j0);
        }
        if (lane == 0) {
            if (A.out_best_dev) A.out_best_dev[b] = best;
            if (A.out_accept_len_dev) A.out_accept_len_dev[b] = acc + 1;
            if (A.out_next_token_dev) A.out_next_token_dev[b] = s_am[last < 0 ? n_rows - 1 : last];
            if (A.cache_len_dev) A.cache_len_dev[b] = start + acc + 1;
            P.kv_start[b] = start;
        }
        // publish: requests that really move rows append their move record {request, accept_len, start, first
        // KV_GROUP source rows} to the compact active list of phase 2
        moved = __reduce_add_sync(SAMD_FULL, moved);
        if (P.n_items2 > 0) {
            int slot = 0;
            if (lane == 0 && moved > 0) slot = atomicAdd(&P.counters[CN_ACTIVE], 1);
            slot = __shfl_sync(SAMD_FULL, slot, 0);
            start = __shfl_sync(SAMD_FULL, start, 0);
            if (moved > 0) {
                int *rec = P.active + (size_t)slot * KV_REC;
                if (lane == 0) rec[0] = b, rec[1] = acc + 1, rec[2] = start;
                if (lane < KV_GROUP) rec[3 + lane] = lane <= acc ? ix0 : lane;
            }
            __syncwarp();
            if (lane == 0) {
                __threadfence();
                if (P.overlap) {
                    // the record (and the outputs phase 2 reads) first, then its flag, then the count of finished walks
                    if (moved > 0) *reinterpret_cast<volatile int *>(&P.act_flag[slot]) = epoch;
                    __threadfence();
                    atomicAdd(&P.counters[CN_WALKS], 1);
                } else if (atomicAdd(&P.counters[CN_ARRIVE_B], 1) == A.batch - 1) {  // barrier B: every walk is published
                    P.counters[CN_ARRIVE_B] = 0;
                    __threadfence();
                    *reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_B]) = epoch;
                }
            }
        }
        if (P.overlap && lane == 0) P.req_done[b] = 0;          // re-armed for the next launch
        __syncwarp();
        if (P.overlap == 2 && P.n_items2 > 0 && moved > 0) {
            // The source rows of this request's moves are known NOW, long before the row moves run (after the last
            // walk): request them into L2 - every 128-byte line of every (tensor, head, row) - so that phase 2 reads hit L2
            // (cp.async.bulk.prefetch.L2 takes a warp-uniform address: 10 k of them per request would be issued one
            // by one; the per-lane prefetch covers 32 rows per instruction) (the 42 MB of config c4 fit three times) instead of scattered DRAM rows.
            const int pairs = A.n_kv * A.n_heads;
            int sj[KV_GROUP];
#pragma unroll
            for (int j = 0; j < KV_GROUP; ++j) {
                const int v = __shfl_sync(SAMD_FULL, ix0, j);
                sj[j] = (j >= 1 && j <= acc && v != j && v >= 0) ? v : -1;
            }
            const int lines = (A.row_bytes + 127) >> 7;
            for (int w = lane; w < pairs; w += 32) {
                const int kv = w / A.n_heads, hd = w - kv * A.n_heads;
                const char *hb = reinterpret_cast<const char *>(__ldg(reinterpret_cast<const unsigned long long *>(A.kv_ptrs_dev) + kv)) +
                                 (size_t)b * A.kv_batch_stride + (size_t)hd * A.kv_head_stride;
#pragma unroll
                for (int j = 1; j < KV_GROUP; ++j)
                    if (sj[j] >= 0)
                        for (int l = 0; l < lines; ++l)
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(hb + (size_t)(start + sj[j]) * A.kv_pos_stride + ((size_t)l << 7)));
            }
        }
    };

    int arrived = 0;                                           // lane 0: items of cur.b reported so far (overlapped flow)
    // ------------------------------ phase 1: row argmax -----------------------------------
    // Items (row chunks) are handed out dynamically - the first one per warp is its own index, the rest come from
    // a counter: measured on B200, equal static shares finish between 27 and 50 us after launch (the memory system
    // is not fair between SMs), so fast warps must be able to take more.  Nothing in the item loop waits on a
    // round trip other than the logits themselves: the result is a fire-and-forget 64-bit max, the next item index
    // is requested one item ahead, and the first vector group of the NEXT item is requested before the current
    // item's last group is folded.
    {
        constexpr bool k16 = kDtype != SAMD_DTYPE_FP32;
        constexpr int G = UNROLL / 2;
        const uint32_t ninf = kDtype == SAMD_DTYPE_BF16 ? 0xFF80FF80u : 0xFC00FC00u;
        const bool vec16 = k16 && P.vec_ok;
        uint4 xa[G], xb[G];
        // only the first p1 warps stream logits (the launch sizes p1 so that the items divide evenly among them, see
        // samd_verify_compact); the others go straight to the barrier and join the row moves
        const int p1 = P.p1_warps;
        Item cur = decode_item(P, gwarp < p1 ? gwarp : P.n_items1), nx;
        int queue = gwarp % N_QUEUES;                           // lane 0's view is the one that counts
        bool stolen = false;
        if constexpr (!kTopK && k16) {
            if (P.tma) {
                // ---- bulk-copy staged stream.  A group = 32 x G consecutive 16-byte vectors (2 KB) of the item; lane 0 asks
                // the copy engine for it - one instruction, completion on the stage's mbarrier - TMA_STAGES groups ahead of
                // the fold, across item boundaries; the warp reads a landed group out of shared memory (conflict-free
                // 128-bit loads) into the registers fold_group works on.  What is in flight no longer lives in registers:
                // 8 KB per warp instead of 2-4, which is what the stream was short of (it ran at the rate of its slowest
                // warps' round trips, not at the DRAM's).
                constexpr int GV = 32 * G;
                uint4 *ring = reinterpret_cast<uint4 *>(reinterpret_cast<unsigned char *>(s_am_all) + P.ring_off) + (size_t)warp * TMA_STAGES * GV;
                unsigned long long *bars = reinterpret_cast<unsigned long long *>(
                                               reinterpret_cast<unsigned char *>(s_am_all) + P.ring_off + (size_t)VW * TMA_STAGES * GV * 16) + warp * TMA_STAGES;
                if (lane == 0)
                    for (int st = 0; st < TMA_STAGES; ++st) mbar_init(&bars[st], 1);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                Item pit = cur;                                 // the item the producer is issuing from
                int pv = 0, pstage = 0, cstage = 0, inflight = 0;
                uint32_t phases = 0;
                auto claim_next = [&]() {                       // blocking claim of the next item (lane 0's atomics)
                    int nxt = 0;
                    if (lane == 0) {
                        nxt = p1 + atomicAdd(&P.counters[CN_QUEUES + queue * QUEUE_STRIDE], 1) * N_QUEUES + queue;
                        if (nxt >= P.n_items1 && !stolen) {
                            stolen = true;
                            queue = (queue + N_QUEUES / 2) % N_QUEUES;
                            nxt = p1 + atomicAdd(&P.counters[CN_QUEUES + queue * QUEUE_STRIDE], 1) * N_QUEUES + queue;
                        }
                    }
                    return decode_item(P, __shfl_sync(SAMD_FULL, nxt, 0));
                };
                auto produce = [&]() {                          // issue the next group, if there is one
                    if (pit.item >= P.n_items1) return;
                    const int nvec = pit.len >> 3;
                    const int nv = min(GV, nvec - pv);
                    if (lane == 0) {
                        mbar_expect_tx(&bars[pstage], (uint32_t)nv * 16u);
                        bulk_g2s(ring + (size_t)pstage * GV, reinterpret_cast<const uint4 *>(logits + item_offset(P, pit)) + pv,
                                 (uint32_t)nv * 16u, &bars[pstage]);
                    }
                    pv += GV;
                    pstage = (pstage + 1) % TMA_STAGES;
                    ++inflight;
                    if (pv >= nvec) {                           // the item is fully requested: on to the next one
                        nx = claim_next();
                        pit = nx;
                        pv = 0;
                    }
                };
                for (int st = 0; st < TMA_STAGES; ++st) produce();
                while (cur.item < P.n_items1) {
                    const int e0 = cur.e0, len = cur.len;
                    const int nvec = len >> 3;
                    const Item mine = cur;
                    uint32_t best_key = 0, best_idx = 0;
                    for (int v0 = 0; v0 < nvec; v0 += GV) {
                        mbar_wait(&bars[cstage], (phases >> cstage) & 1u);
                        phases ^= 1u << cstage;
                        const uint4 *sg = ring + (size_t)cstage * GV;
#pragma unroll
                        for (int u = 0; u < G; ++u) {
                            const int vi = v0 + u * 32 + lane;
                            xa[u] = vi < nvec ? sg[u * 32 + lane] : make_uint4(ninf, ninf, ninf, ninf);
                        }
                        cstage = (cstage + 1) % TMA_STAGES;
                        --inflight;
                        // fold first: its warp-wide reduction consumes every lane's vectors, so all reads of the stage are
                        // complete before lane 0 hands the stage back to the copy engine
                        fold_group<kDtype, G>(xa, v0, nvec, lane, e0, best_key, best_idx);
                        __syncwarp();
                        produce();
                    }
                    const uint16_t *row = logits + item_offset(P, mine);
                    const int tail = nvec << 3;
                    if (len - tail > 0) {                       // < 8 trailing elements, all later than the vectors
                        const uint32_t ke = lane < len - tail ? orderable16<kDtype>(row[tail + lane]) : 0u;
                        const uint32_t wk = __reduce_max_sync(SAMD_FULL, ke);
                        if (wk > best_key) {
                            best_key = wk;
                            best_idx = (uint32_t)(e0 + tail + __ffs(__ballot_sync(SAMD_FULL, ke == wk)) - 1);
                        }
                    }
                    if (lane == 0) {
                        const unsigned long long pk =
                            best_key ? (((unsigned long long)best_key << 32) | (unsigned long long)(0xFFFFFFFFu - best_idx)) : 0ull;
                        unsigned long long *kp = &P.node_key[(size_t)mine.b * P.max_nodes + mine.t];
                        if (C == 1) *reinterpret_cast<volatile unsigned long long *>(kp) = pk;
                        else atomicMax(kp, pk);
                    }
                    // the producer finished this item at least one group ago (an item has more groups than the ring has
                    // stages), so `nx` is the item that follows it
                    cur = nx;
                }
                cur = decode_item(P, P.n_items1);               // nothing left for the register-staged loop below
            }
        }
        if (vec16 && cur.act)
            load_group<G>(xa, reinterpret_cast<const uint4 *>(logits + item_offset(P, cur)), 0, cur.len >> 3, lane, ninf);
        for (; cur.item < P.n_items1; cur = nx) {
            // (claiming later - one pass before the item is needed - measured slower: 52.4 vs 49.5 us on C4)
            int claim = 0;                                      // requested now, consumed in the item's last pass
            if (lane == 0) claim = atomicAdd(&P.counters[CN_QUEUES + queue * QUEUE_STRIDE], 1);
            bool fetched = false;
            auto fetch_next = [&]() {
                int nxt = 0;
                if (lane == 0) {
                    nxt = p1 + claim * N_QUEUES + queue;
                    if (nxt >= P.n_items1 && !stolen) {         // home queue drained: one try at the opposite queue
                        stolen = true;
                        queue = (queue + N_QUEUES / 2) % N_QUEUES;
                        nxt = p1 + atomicAdd(&P.counters[CN_QUEUES + queue * QUEUE_STRIDE], 1) * N_QUEUES + queue;
                    }
                }
                nx = decode_item(P, __shfl_sync(SAMD_FULL, nxt, 0));
                fetched = true;
                if (vec16 && nx.act)
                    load_group<G>(xa, reinterpret_cast<const uint4 *>(logits + item_offset(P, nx)), 0, nx.len >> 3, lane, ninf);
            };
            if (cur.act) {
                const int e0 = cur.e0, len = cur.len;
                const uint16_t *row = logits + item_offset(P, cur);
                uint32_t best_key = 0, best_idx = 0;
                unsigned long long tk = 0;                      // top-k launches: lanes 0..7 hold the sorted list
                uint32_t thrv = 0, floorv = key_ninf<kDtype>();
                if constexpr (kDtype == SAMD_DTYPE_FP32) {
                    // fp32 logits (the reference's --dtype float32 runs): coalesced scalar loads, per-lane maxima
                    const uint32_t *row32 = reinterpret_cast<const uint32_t *>(A.logits_dev) + item_offset(P, cur);
                    if constexpr (kTopK) {
                        for (int e = 0; e < len; e += 32) {
                            const uint32_t ke = e + lane < len ? orderable32(__ldg(row32 + e + lane)) : 0u;
                            fold_elems_topk<kDtype>(ke, (uint32_t)(e0 + e + lane), tk, thrv, lane);
                        }
                    } else {
#pragma unroll 4
                        for (int e = lane; e < len; e += 32) {
                            const uint32_t ke = orderable32(__ldg(row32 + e));
                            if (ke > best_key) {
                                best_key = ke;
                                best_idx = (uint32_t)(e0 + e);
                            }
                        }
                    }
                } else if (P.vec_ok) {
                    // The running maximum is WARP-uniform: a group of 32 x G vectors is reduced to one key per lane
                    // with packed max instructions, then across lanes with redux.sync; only when the group beats the
                    // running maximum (about ln(#groups) times per row) is the first maximal element located, from
                    // the registers that still hold the group.  The loads of the next half-group are in flight
                    // while this one is folded (xa was requested before this item began).
                    const uint4 *v4 = reinterpret_cast<const uint4 *>(row);
                    const int nvec = len >> 3;
                    if constexpr (kTopK) {
                        if (nvec >= 32 * G) floorv = topk_floor<kDtype, G>(xa, lane);   // a full first group
                    }
                    for (int v0 = 0; v0 < nvec; v0 += 64 * G) {
                        const int v1 = v0 + 32 * G;
                        if (v1 < nvec) load_group<G>(xb, v4, v1, nvec, lane, ninf);
                        if constexpr (kTopK) fold_group_topk<kDtype, G>(xa, v0, nvec, lane, e0, tk, thrv, floorv);
                        else fold_group<kDtype, G>(xa, v0, nvec, lane, e0, best_key, best_idx);
                        if (v1 + 32 * G < nvec) load_group<G>(xa, v4, v1 + 32 * G, nvec, lane, ninf);
                        else fetch_next();                      // last pass: xa is free, start on the next item
                        if (v1 < nvec) {
                            if constexpr (kTopK) fold_group_topk<kDtype, G>(xb, v1, nvec, lane, e0, tk, thrv, floorv);
                            else fold_group<kDtype, G>(xb, v1, nvec, lane, e0, best_key, best_idx);
                        }
                    }
                    const int tail = nvec << 3;
                    if (len - tail > 0) {                      // < 8 trailing elements, all later than the vectors
                        const uint32_t ke = lane < len - tail ? orderable16<kDtype>(row[tail + lane]) : 0u;
                        if constexpr (kTopK) {
                            fold_elems_topk<kDtype>(ke, (uint32_t)(e0 + tail + lane), tk, thrv, lane);
                        } else {
                            const uint32_t wk = __reduce_max_sync(SAMD_FULL, ke);
                            if (wk > best_key) {
                                best_key = wk;
                                best_idx = (uint32_t)(e0 + tail + __ffs(__ballot_sync(SAMD_FULL, ke == wk)) - 1);
                            }
                        }
                    }
                } else {
                    if constexpr (kTopK) {
                        for (int e = 0; e < len; e += 32) {
                            const uint32_t ke = e + lane < len ? orderable16<kDtype>(row[e + lane]) : 0u;
                            fold_elems_topk<kDtype>(ke, (uint32_t)(e0 + e + lane), tk, thrv, lane);
                        }
                    } else {
                        for (int e = lane; e < len; e += 32) {
                            const uint32_t ke = orderable16<kDtype>(row[e]);
                            if (ke > best_key) {
                                best_key = ke;
                                best_idx = (uint32_t)(e0 + e);
                            }
                        }
                    }
                }
                unsigned long long pk;
                if constexpr (kTopK) {
                    if (lane < TOPK) P.topk_part[(size_t)cur.item * TOPK + lane] = tk;
                    pk = __shfl_sync(SAMD_FULL, tk, 0);         // the argmax is the head of the list ...
                    if (pk == 0 && len > 0)                     // ... unless the whole chunk is -inf: its first element
                        pk = ((unsigned long long)key_ninf<kDtype>() << 32) | (0xFFFFFFFFu - (uint32_t)e0);
                } else {
                    pk = best_key ? (((unsigned long long)best_key << 32) | (unsigned long long)(0xFFFFFFFFu - best_idx)) : 0ull;
                    if (!vec16) {                               // per-lane maxima: combine (the vector path is warp-uniform)
#pragma unroll
                        for (int o = 16; o; o >>= 1) {
                            const unsigned long long other = __shfl_xor_sync(SAMD_FULL, pk, o);
                            pk = other > pk ? other : pk;
                        }
                    }
                }
                if (lane == 0) {
                    unsigned long long *kp = &P.node_key[(size_t)cur.b * P.max_nodes + cur.t];
                    if constexpr (!kTopK) {
                        if (P.overlap) {
                            // The maximum comes back (so it HAS been performed at L2), and only then is the request's
                            // arrival counted - the add's operand depends on the returned value.  Whoever counts the
                            // request's last item therefore finds every row maximum in L2 without any fence.
                            const unsigned long long old = atomicMax(kp, pk);
                            int dep;
                            asm volatile("and.b32 %0, %1, 0;" : "=r"(dep) : "r"((int)old));
                            arrived = atomicAdd(&P.req_done[cur.b], 1 + dep) + 1;
                        } else if (C == 1) *reinterpret_cast<volatile unsigned long long *>(kp) = pk;
                        else atomicMax(kp, pk);
                    } else {
                        if (C == 1) *reinterpret_cast<volatile unsigned long long *>(kp) = pk;
                        else atomicMax(kp, pk);
                    }
                }
            } else {
                if constexpr (kTopK) {
                    if (lane < TOPK) P.topk_part[(size_t)cur.item * TOPK + lane] = 0;   // dead row: empty list
                } else if (P.overlap && lane == 0) {
                    arrived = atomicAdd(&P.req_done[cur.b], 1) + 1;                     // dead row: it still counts
                }
            }
            if (!fetched) fetch_next();
            if constexpr (!kTopK) {
                if (P.overlap) {
                    // the warp that reports a request's last item walks it at once (the next item's first loads are
                    // already in flight): its row moves can start while the rest of the logits still stream
                    const int done_b = __shfl_sync(SAMD_FULL, arrived == T * C ? cur.b : -1, 0);
                    arrived = 0;
                    if (done_b >= 0) walk_request(done_b);
                }
            }
        }
    }
    if (dbg && lane == 0) dbg[1] = samd_globaltimer();

    // ------------------------------ barrier A: every row maximum is published -----------------
    if (!P.overlap) {
    if (lane == 0) __threadfence();                            // this warp's keys, before the CTA arrives
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&P.counters[CN_ARRIVE_A], 1) == n_ctas - 1) {
            P.counters[CN_ARRIVE_A] = 0;
            __threadfence();
            *reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_A]) = epoch;
        }
    }

    if constexpr (kTopK) {                                      // every warp merges rows: the whole CTA waits for A
        if (threadIdx.x == 0) {
            while (*reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_A]) != epoch) __nanosleep(100);
            __threadfence();
        }
        __syncthreads();
    }
    // ------------------------------ phase 1b: path walks (samd/utils.py:127-141) ---------------
    // one warp per request, spread over the SMs (warp 0 of CTA b for the first n_ctas requests); CTAs with neither
    // a walk nor row moves to do leave right after arriving
    if (gwarp < A.batch) {
        if (lane == 0) {
            while (*reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_A]) != epoch) __nanosleep(100);
            __threadfence();
        }
        __syncwarp();
    }
    }   // !P.overlap
    if (!P.overlap)
        for (int b = gwarp; b < A.batch; b += n_warps) walk_request(b);

    // ------------------------------ phase 1c: per-row top-8 (token_recycle.py:36-47) ----------
    // The chunks' lists are merged row by row (rows strided over every warp); the row that comes last in (request,
    // node) order among those feeding the same token claims that token's table entry (the reference overwrites
    // cache[token] in zip order), and writes it once every claim is in (barrier C, waited for after the row moves).
    if constexpr (kTopK) {
        const int n_rows_total = A.batch * T;
        for (int row = gwarp; row < n_rows_total; row += n_warps) {
            const int b = row / T, tt = row - b * T;
            const bool live = tt < (A.n_nodes_dev ? A.n_nodes_dev[b] : T);
            unsigned long long tk = 0;
            uint32_t thrv = 0;
            if (live) {
                const unsigned long long *part = P.topk_part + (size_t)row * C * TOPK;
                for (int c0 = 0; c0 < C * TOPK; c0 += 32) {
                    unsigned long long c = c0 + lane < C * TOPK ? __ldcg(part + c0 + lane) : 0ull;
                    while (true) {
                        unsigned long long m = c;
#pragma unroll
                        for (int o = 16; o; o >>= 1) {
                            const unsigned long long other = __shfl_xor_sync(SAMD_FULL, m, o);
                            m = other > m ? other : m;
                        }
                        if (m == 0 || m <= __shfl_sync(SAMD_FULL, tk, TOPK - 1)) break;
                        topk_insert(m, tk, thrv, lane);
                        if (c == m) c = 0;                      // composites are unique (they carry the index)
                    }
                }
                // fewer than 8 elements above -inf: completed with the lowest-index -inf elements
                int have = __popc(__ballot_sync(SAMD_FULL, lane < TOPK && tk != 0));
                for (int e = 0; e < A.vocab && have < TOPK; e += 32) {
                    uint32_t ke = 0;
                    if (e + lane < A.vocab) {
                        const size_t off = (size_t)b * A.batch_stride + (size_t)tt * A.row_stride + e + lane;
                        if constexpr (kDtype == SAMD_DTYPE_FP32) ke = orderable32(reinterpret_cast<const uint32_t *>(A.logits_dev)[off]);
                        else ke = orderable16<kDtype>(logits[off]);
                    }
                    unsigned bal = __ballot_sync(SAMD_FULL, ke == key_ninf<kDtype>());
                    while (bal && have < TOPK) {
                        const uint32_t idx = (uint32_t)(e + __ffs(bal) - 1);
                        if (lane == have) tk = ((unsigned long long)key_ninf<kDtype>() << 32) | (0xFFFFFFFFu - idx);
                        ++have;
                        bal &= bal - 1;
                    }
                }
            }
            if (lane < TOPK && A.out_topk_dev) A.out_topk_dev[(size_t)row * TOPK + lane] = tk ? (int)(0xFFFFFFFFu - (uint32_t)tk) : -1;
            if (A.recycle_table_dev && live && lane == 0) {
                const int tok = A.tree_tokens_dev[row];
                if (tok >= 0 && tok < A.vocab) atomicMax(&A.recycle_owner_dev[tok], row);
            }
        }
        if (A.recycle_table_dev) {                              // barrier C, arrival
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                if (atomicAdd(&P.counters[CN_ARRIVE_C], 1) == n_ctas - 1) {
                    P.counters[CN_ARRIVE_C] = 0;
                    __threadfence();
                    *reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_C]) = epoch;
                }
            }
        }
    }

    // ------------------------------ phase 2: KV row moves ---------------------------------
    // The moved rows of the active requests are flattened into 16-byte units and strided over every lane of the
    // grid.  (Dedicating a quarter of the CTAs to row moves that overlap the logits stream was measured slower,
    // 111 vs 90 us on C4: the moves are bound by DRAM row activations and steal DRAM cycles from the stream.)
    if (P.n_items2 > 0 && P.overlap == 1) {
        // Overlapped flow: a warp that finds no more logits to stream takes TICKETS - (move record, chunk of its 16-byte
        // units) - and waits only for that record's flag, so the rows of the requests that completed first are moved
        // while the later ones are still being streamed and walked.  A ticket beyond the last record ends the warp
        // once every walk has reported.
        const int cols = A.row_bytes >> 4;
        const int per_tensor = A.n_heads * cols;
        const int per_req = A.n_kv * per_tensor;
        constexpr int UNITS = 256;                             // 16-byte units (x accepted rows) per ticket: 8 passes of a warp
        const int n_ch = (per_req + UNITS - 1) / UNITS;
        int t = 0;
        if (lane == 0) t = atomicAdd(&P.counters[CN_TICKET], 1);
        while (true) {
            t = __shfl_sync(SAMD_FULL, t, 0);
            const int a_i = t / n_ch, ch = t - a_i * n_ch;
            if (a_i >= A.batch) break;                          // beyond any possible record
            int have = 0;
            if (lane == 0) {
                t = atomicAdd(&P.counters[CN_TICKET], 1);       // the next ticket is requested one ahead
                unsigned ns = 200;
                for (int spin = 0;; ++spin) {
                    if (*reinterpret_cast<volatile int *>(&P.act_flag[a_i]) == epoch) {
                        have = 1;
                        break;
                    }
                    if ((spin & 3) == 3 && *reinterpret_cast<volatile int *>(&P.counters[CN_WALKS]) == A.batch) {
                        have = *reinterpret_cast<volatile int *>(&P.act_flag[a_i]) == epoch;   // flags precede the count
                        break;
                    }
                    __nanosleep(ns);                            // (thousands of warps may be waiting: back off)
                    if (ns < 3200) ns *= 2;
                }
                __threadfence();
            }
            have = __shfl_sync(SAMD_FULL, have, 0);
            if (!have) break;                                   // every walk has reported and there is no such record
            const int *m = P.active + (size_t)a_i * KV_REC;
            const int b = __ldcg(m), acc1 = __ldcg(m + 1), start = __ldcg(m + 2);
            int src0[KV_GROUP];
#pragma unroll
            for (int q = 0; q < KV_GROUP; ++q) src0[q] = __ldcg(m + 3 + q);
            const int u_end = min(per_req, (ch + 1) * UNITS);
            for (int unit = ch * UNITS + lane; unit < u_end; unit += 32) {
                const int kv = unit / per_tensor;
                const int w = unit - kv * per_tensor;
                const int hd = w / cols, col = w - hd * cols;
                char *hb = reinterpret_cast<char *>(__ldg(reinterpret_cast<const unsigned long long *>(A.kv_ptrs_dev) + kv)) +
                           (size_t)b * A.kv_batch_stride + (size_t)hd * A.kv_head_stride + ((size_t)col << 4);
                for (int j0 = 0; j0 < acc1; j0 += KV_GROUP) {
                    uint4 val[KV_GROUP];
                    int src[KV_GROUP];
#pragma unroll
                    for (int q = 0; q < KV_GROUP; ++q)
                        src[q] = j0 == 0 ? src0[q] : ((j0 + q < acc1) ? __ldcg(A.out_indices_dev + (size_t)b * A.depth + j0 + q) : j0 + q);
#pragma unroll
                    for (int q = 0; q < KV_GROUP; ++q)
                        if (src[q] != j0 + q) val[q] = *reinterpret_cast<const uint4 *>(hb + (size_t)(start + src[q]) * A.kv_pos_stride);
#pragma unroll
                    for (int q = 0; q < KV_GROUP; ++q)
                        if (src[q] != j0 + q) *reinterpret_cast<uint4 *>(hb + (size_t)(start + j0 + q) * A.kv_pos_stride) = val[q];
                }
            }
        }
    } else if (P.n_items2 > 0) {
        const int cols = A.row_bytes >> 4;                      // 16-byte columns per (head,row)
        const int per_tensor = A.n_heads * cols;
        const long long per_req = (long long)A.n_kv * per_tensor;
        constexpr int MW = KV_REC;
        int *s_meta = s_am_all + VW * 2 * T;
        __syncthreads();
        if (threadIdx.x == 0) {                                 // one poller per CTA, plain loads, backoff
            if (P.overlap) while (*reinterpret_cast<volatile int *>(&P.counters[CN_WALKS]) != A.batch) __nanosleep(200);
            else while (*reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_B]) != epoch) __nanosleep(200);
            __threadfence();
        }
        __syncthreads();
        const int n_active = __ldcg(&P.counters[CN_ACTIVE]);
        const int *active = P.active;
        const long long total = per_req * n_active;
        // stage the move records in shared memory: no dependent metadata loads in the copy loop
        const int staged = min(n_active, P.stage_cap);
        for (int i = threadIdx.x; i < staged * MW; i += VT) s_meta[i] = __ldcg(active + i);
        __syncthreads();
        // (more loads in flight per lane - 4 units x 2 rows - was measured: 98 vs 89 us; the row moves are
        // bound by scattered 256-byte DRAM accesses with read/write turnarounds, not by latency)
        for (long long u = (long long)gwarp * 32 + lane; u < total; u += (long long)n_warps * 32) {
            const int a_i = (int)(u / per_req);
            const int unit = (int)(u - (long long)a_i * per_req);
            int b, acc1, start;
            int src[KV_GROUP];
            if (a_i < staged) {
                const int *m = s_meta + a_i * MW;
                b = m[0];
                acc1 = m[1];
                start = m[2];
#pragma unroll
                for (int q = 0; q < KV_GROUP; ++q) src[q] = m[3 + q];
            } else {
                const int *m = active + (size_t)a_i * MW;
                b = __ldcg(m);
                acc1 = __ldcg(m + 1);
                start = __ldcg(m + 2);
#pragma unroll
                for (int q = 0; q < KV_GROUP; ++q) src[q] = __ldcg(m + 3 + q);
            }
            const int kv = unit / per_tensor;
            const int w = unit - kv * per_tensor;
            const int hd = w / cols, col = w - hd * cols;
            char *hb = reinterpret_cast<char *>(__ldg(reinterpret_cast<const unsigned long long *>(A.kv_ptrs_dev) + kv)) +
                       (size_t)b * A.kv_batch_stride + (size_t)hd * A.kv_head_stride + ((size_t)col << 4);
            for (int j0 = 0; j0 < acc1; j0 += KV_GROUP) {
                uint4 val[KV_GROUP];
                if (j0 > 0) {
#pragma unroll
                    for (int q = 0; q < KV_GROUP; ++q)
                        src[q] = (j0 + q < acc1) ? __ldcg(A.out_indices_dev + (size_t)b * A.depth + j0 + q) : j0 + q;
                }
#pragma unroll
                for (int q = 0; q < KV_GROUP; ++q)
                    if (src[q] != j0 + q) val[q] = *reinterpret_cast<const uint4 *>(hb + (size_t)(start + src[q]) * A.kv_pos_stride);
#pragma unroll
                for (int q = 0; q < KV_GROUP; ++q)
                    if (src[q] != j0 + q) *reinterpret_cast<uint4 *>(hb + (size_t)(start + j0 + q) * A.kv_pos_stride) = val[q];
            }
        }
    }
    if constexpr (kTopK) {
        if (A.recycle_table_dev) {                              // barrier C, wait; then the owners write their entries
            __syncthreads();
            if (threadIdx.x == 0) {
                while (*reinterpret_cast<volatile int *>(&P.counters[CN_FLAG_C]) != epoch) __nanosleep(100);
                __threadfence();
            }
            __syncthreads();
            const int n_rows_total = A.batch * T;
            for (int row = gwarp; row < n_rows_total; row += n_warps) {
                const int b = row / T, tt = row - b * T;
                if (tt >= (A.n_nodes_dev ? A.n_nodes_dev[b] : T)) continue;
                const int tok = A.tree_tokens_dev[row];
                if (tok < 0 || tok >= A.vocab || __ldcg(&A.recycle_owner_dev[tok]) != row) continue;
                if (lane < TOPK) A.recycle_table_dev[(size_t)tok * TOPK + lane] = __ldcg(&A.out_topk_dev[(size_t)row * TOPK + lane]);
                __syncwarp();
                if (lane == 0) A.recycle_owner_dev[tok] = -1;   // re-armed for the next launch
            }
        }
    }
    if (dbg && lane == 0) dbg[2] = samd_globaltimer();
    // last CTA out: re-arm the work and active counters and bump the device-side epoch (every CTA read it before it
    // could change)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&P.counters[CN_EXIT], 1) == n_ctas - 1) {
            P.counters[CN_EXIT] = 0;
            P.counters[CN_ACTIVE] = 0;
            P.counters[CN_TICKET] = 0;
            P.counters[CN_WALKS] = 0;
            for (int q = 0; q < N_QUEUES; ++q) P.counters[CN_QUEUES + q * QUEUE_STRIDE] = 0;
            __threadfence();
            *reinterpret_cast<volatile int *>(&P.counters[CN_EPOCH]) = epoch;
        }
    }
}

extern "C" int samd_verify_create(int max_batch, int max_nodes, samd_verify_t *out) {
    SAMD_REQUIRE(max_batch > 0 && max_nodes > 0 && out, "samd_verify_create: bad arguments");
    samd_verify_s *h = new samd_verify_s();
    h->max_batch = max_batch;
    h->max_nodes = max_nodes;
    for (int &o : h->occ_per_sm) o = 0;
    SAMD_CUDA(cudaGetDevice(&h->device));
    SAMD_CUDA(cudaDeviceGetAttribute(&h->n_sms, cudaDevAttrMultiProcessorCount, h->device));
    SAMD_CUDA(cudaMalloc(&h->node_key, (size_t)max_batch * max_nodes * sizeof(unsigned long long)));
    SAMD_CUDA(cudaMalloc(&h->active, (size_t)max_batch * KV_REC * sizeof(int)));
    SAMD_CUDA(cudaMalloc(&h->counters, CN_WORDS * sizeof(int)));
    SAMD_CUDA(cudaMalloc(&h->kv_start, (size_t)max_batch * sizeof(int)));
    SAMD_CUDA(cudaMalloc(&h->req_done, (size_t)max_batch * sizeof(int)));
    SAMD_CUDA(cudaMalloc(&h->act_flag, (size_t)max_batch * sizeof(int)));
    SAMD_CUDA(cudaMemset(h->req_done, 0, (size_t)max_batch * sizeof(int)));
    SAMD_CUDA(cudaMemset(h->act_flag, 0, (size_t)max_batch * sizeof(int)));
    h->topk_items = std::max<long long>((long long)max_batch * max_nodes * 16, 32768);
    SAMD_CUDA(cudaMalloc(&h->topk_part, (size_t)h->topk_items * 8 * sizeof(unsigned long long)));
    SAMD_CUDA(cudaMemset(h->node_key, 0, (size_t)max_batch * max_nodes * sizeof(unsigned long long)));
    SAMD_CUDA(cudaMemset(h->active, 0, (size_t)max_batch * KV_REC * sizeof(int)));
    SAMD_CUDA(cudaMemset(h->counters, 0, CN_WORDS * sizeof(int)));
    SAMD_CUDA(cudaMemset(h->kv_start, 0, (size_t)max_batch * sizeof(int)));
    SAMD_CUDA(cudaDeviceSynchronize());
    *out = h;
    return 0;
}

extern "C" int samd_verify_destroy(samd_verify_t h) {
    if (!h) return 0;
    cudaFree(h->node_key);
    cudaFree(h->active);
    cudaFree(h->counters);
    cudaFree(h->kv_start);
    cudaFree(h->req_done);
    cudaFree(h->act_flag);
    cudaFree(h->topk_part);
    delete h;
    return 0;
}

static int g_chunk_override = 0;
static int g_min_chunk = 2048;
static int g_overlap = 0;
static int g_even_items = 1;
static int g_tma = 0;
extern "C" void samd_verify_set_tma(int on) { g_tma = on; }
extern "C" void samd_verify_set_even_items(int on) { g_even_items = on; }
extern "C" void samd_verify_set_overlap(int on) { g_overlap = on; }
static unsigned long long *g_dbg_times = nullptr;
extern "C" void samd_verify_set_debug_times(uint64_t *times_dev) { g_dbg_times = (unsigned long long *)times_dev; }
extern "C" void samd_verify_set_chunk(int elements) { g_chunk_override = elements; }

extern "C" int samd_verify_compact(samd_verify_t h, const samd_verify_args *a, void *stream) {
    SAMD_REQUIRE(h && a, "samd_verify_compact: bad arguments");
    SAMD_REQUIRE(a->logits_dev && a->tree_tokens_dev, "samd_verify_compact: logits and tree tokens are required");
    SAMD_REQUIRE(a->batch > 0 && a->batch <= h->max_batch, "samd_verify_compact: batch exceeds scratch capacity");
    SAMD_REQUIRE(a->n_nodes > 0 && a->n_nodes <= h->max_nodes, "samd_verify_compact: n_nodes exceeds scratch capacity");
    SAMD_REQUIRE(a->vocab > 0, "samd_verify_compact: bad vocab");
    SAMD_REQUIRE(a->dtype == SAMD_DTYPE_BF16 || a->dtype == SAMD_DTYPE_FP16 || a->dtype == SAMD_DTYPE_FP32,
                 "samd_verify_compact: bad dtype");
    SAMD_REQUIRE(!a->retrieve_dev || (a->n_paths > 0 && a->n_paths < 65535 && a->depth > 0 && a->depth < 65535),
                 "samd_verify_compact: bad retrieve table shape");
    const bool move = a->move_kv && a->kv_ptrs_dev && a->retrieve_dev;
    if (move) {
        SAMD_REQUIRE(a->out_accept_len_dev && a->out_indices_dev, "samd_verify_compact: KV moves need accept_len and indices outputs");
        SAMD_REQUIRE(a->row_bytes > 0 && a->row_bytes % 16 == 0 && a->kv_pos_stride % 16 == 0 && a->kv_head_stride % 16 == 0 &&
                         a->kv_batch_stride % 16 == 0,
                     "samd_verify_compact: KV rows must be 16-byte aligned");
        SAMD_REQUIRE(a->n_kv > 0 && a->n_heads > 0, "samd_verify_compact: bad KV shape");
    }
    VerifyParams P;
    P.a = *a;
    P.node_key = h->node_key;
    P.active = h->active;
    P.counters = h->counters;
    P.max_batch = h->max_batch;
    P.kv_start = h->kv_start;
    P.req_done = h->req_done;
    P.act_flag = h->act_flag;
    P.dbg_times = g_dbg_times;
    P.max_nodes = h->max_nodes;
    P.stage_cap = move ? std::min(a->batch, 512) : 0;
    size_t smem = ((size_t)VW * 2 * a->n_nodes + (size_t)P.stage_cap * (3 + KV_GROUP)) * sizeof(int);
    const bool topk = a->out_topk_dev != nullptr;
    P.overlap = topk ? 0 : g_overlap;
    P.tma = 0;
    P.ring_off = 0;
    SAMD_REQUIRE(!a->recycle_table_dev || (topk && a->recycle_owner_dev),
                 "samd_verify_compact: a recycle table needs out_topk_dev and recycle_owner_dev");
    SAMD_REQUIRE(!topk || a->vocab >= TOPK, "samd_verify_compact: top-8 needs a vocabulary of at least 8");
    P.topk_part = h->topk_part;
    auto kern = a->dtype == SAMD_DTYPE_BF16   ? (topk ? verify_compact_kernel<SAMD_DTYPE_BF16, true> : verify_compact_kernel<SAMD_DTYPE_BF16, false>)
                : a->dtype == SAMD_DTYPE_FP16 ? (topk ? verify_compact_kernel<SAMD_DTYPE_FP16, true> : verify_compact_kernel<SAMD_DTYPE_FP16, false>)
                                              : (topk ? verify_compact_kernel<SAMD_DTYPE_FP32, true> : verify_compact_kernel<SAMD_DTYPE_FP32, false>);
    // Bulk-copy staging of the logits stream (16-bit logits, no top-8, no dead rows, barrier flow, aligned rows, a
    // vocabulary large enough for items of several groups): every warp gets a ring of TMA_STAGES 2 KB stages + mbarriers
    P.vec_ok = ((uintptr_t)a->logits_dev % 16 == 0) && (a->batch_stride % 8 == 0) && (a->row_stride % 8 == 0);
    const bool tma_ok = g_tma && !topk && a->dtype != SAMD_DTYPE_FP32 && P.vec_ok && !P.overlap && !a->n_nodes_dev && a->vocab >= 16384;
    if (tma_ok) {
        P.ring_off = (int)((smem + 127) & ~(size_t)127);
        smem = (size_t)P.ring_off + (size_t)VW * TMA_STAGES * (32 * (UNROLL / 2)) * 16 + (size_t)VW * TMA_STAGES * 8;
        P.tma = 1;
    }
    if (smem > 48 * 1024) {
        // large path tables (eval_posterior verifies P*D rows as nodes): beyond 48 KB the kernel has to opt in
        SAMD_REQUIRE(smem <= 200 * 1024, "samd_verify_compact: n_nodes too large for the per-warp node tables in shared memory");
        SAMD_CUDA(cudaFuncSetAttribute((const void *)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    int per_sm = h->occ_per_sm[a->dtype + (topk ? 3 : 0)];
    if (per_sm <= 0 || smem > 8192) {                           // cached for the common (small) shared-memory sizes
        SAMD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, VT, smem > 8192 ? smem : 8192));
        if (smem <= 8192) h->occ_per_sm[a->dtype + (topk ? 3 : 0)] = per_sm;
    }
    SAMD_REQUIRE(per_sm > 0, "samd_verify_compact: kernel does not fit on an SM");
    // persistent grid: every CTA must be resident (the kernel has grid-wide barriers)
    const long long rows = (long long)a->batch * a->n_nodes;
    const long long resident_warps = (long long)h->n_sms * per_sm * VW;
    // Items are handed out dynamically.  Measured on C4 (uniform chunks): 16000 elements 50.0 us, 8192 51.4, 4000
    // 54.3, 2000 67.4, whole rows 53.7 - an item switch costs about half a microsecond of issue latency, so chunks
    // are about 16k elements unless the launch is too small to give every resident warp one.
    int chunks = std::max(1, (a->vocab + 8192) / 16384);
    while (rows * chunks < resident_warps && a->vocab / (chunks * 2) >= g_min_chunk) chunks *= 2;
    if (g_chunk_override > 0) chunks = (a->vocab + g_chunk_override - 1) / g_chunk_override;
    const int chunk = ((a->vocab + chunks - 1) / chunks + 7) & ~7;
    P.chunk = chunk;
    P.chunks_per_row = (a->vocab + chunk - 1) / chunk;
    P.n_items1 = (int)rows * P.chunks_per_row;
    SAMD_REQUIRE(!topk || P.n_items1 <= h->topk_items, "samd_verify_compact: top-8 scratch too small for this shape");
    P.n_items2 = move ? a->batch * a->n_kv : 0;
    // the staged stream runs TMA_STAGES groups ahead, across ONE item boundary: every item must hold more groups than that
    if (P.tma && a->vocab - (P.chunks_per_row - 1) * chunk < (TMA_STAGES + 1) * 32 * (UNROLL / 2) * 8) P.tma = 0;
    // One warp per item up to the resident grid.  With row moves, a small batch keeps a small grid too (every CTA
    // takes part in the barriers, whose cost grows with their number: 20.6 -> 19.1 us per launch at batch 1) as long as
    // each moved request still finds about 32 CTAs' worth of lanes for its 16-byte units.
    const long long full = std::max<long long>(1, (long long)h->n_sms * per_sm);
    long long grid = std::min<long long>(full, ((long long)P.n_items1 + VW - 1) / VW);
    if (move) grid = std::max<long long>(grid, std::min<long long>(full, (long long)a->batch * 32));
    grid = std::max<long long>(grid, 1);
    // Phase-1 warps.  Every warp streams at about the same rate, so the phase ends when the warps with the most items end:
    // 7808 items over 4736 resident warps means 3072 warps stream two items while 1664 idle through the second half
    // (measured: first items end at 20-24 us, second ones at 37-44).  With p1 = ceil(items / ceil(items / warps)) every
    // streaming warp gets the same number of items (c4: 3904 warps x 2, c5: 4462 x 7) and the rest of the grid waits at
    // the barrier for the row moves.
    {
        const long long w = grid * VW;
        const long long per = std::max<long long>(1, (P.n_items1 + w - 1) / w);
        P.p1_warps = g_even_items ? (int)std::min<long long>(w, (P.n_items1 + per - 1) / per) : (int)w;
    }
    // Cooperative launch: the kernel's barriers need every CTA resident at once, and only a cooperative launch makes
    // the driver guarantee it - two overlapping launches (two handles on two streams) would otherwise each hold part
    // of the machine and wait for the rest forever.
    // (Measured: no cost against a plain launch, 78.8 vs 79.1 us on C4, and it replays inside CUDA graphs.)
    void *kargs[] = {(void *)&P};
    SAMD_CUDA(cudaLaunchCooperativeKernel((const void *)kern, dim3((unsigned)grid), dim3(VT), kargs, smem, (cudaStream_t)stream));
    samd_count_launch();
    return 0;
}

// ---------------------------------------------------------------------------------------
// Stand-alone SamdStaticCache.select_indices (samd/cache.py:118-133) for callers that verify
// elsewhere: same row moves as phase 2 above, indices / accept lengths given by the caller.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(VT) kv_compact_kernel(void *const *kv_ptrs, int n_kv, int n_heads, int row_bytes,
                                                        long long batch_stride, long long head_stride, long long pos_stride,
                                                        const int32_t *indices, int depth, const int32_t *accept_len,
                                                        int32_t *cache_len, int batch, int bump) {
    const int lane = threadIdx.x & 31;
    const int gwarp = (blockIdx.x * VT + threadIdx.x) >> 5;
    const int n_warps = (gridDim.x * VT) >> 5;
    const int cols = row_bytes >> 4;
    const int per_tensor = n_heads * cols;
    for (int item = gwarp; item < batch * n_kv; item += n_warps) {
        const int b = item / n_kv, kv = item % n_kv;
        const int acc1 = accept_len[b];
        const int start = cache_len[b];
        const int32_t *idx = indices + (size_t)b * depth;
        char *base = reinterpret_cast<char *>(kv_ptrs[kv]) + (size_t)b * batch_stride;
        for (int j0 = 0; j0 < acc1; j0 += KV_GROUP) {
            int src[KV_GROUP];
            bool any = false;
#pragma unroll
            for (int u = 0; u < KV_GROUP; ++u) {
                src[u] = (j0 + u < acc1) ? idx[j0 + u] : j0 + u;
                any |= src[u] != j0 + u;
            }
            if (!any) continue;
            for (int w = lane; w < per_tensor; w += 32) {
                const int hd = w / cols, col = w - hd * cols;
                char *hb = base + (size_t)hd * head_stride + ((size_t)col << 4);
                uint4 val[KV_GROUP];
#pragma unroll
                for (int u = 0; u < KV_GROUP; ++u)
                    if (src[u] != j0 + u) val[u] = *reinterpret_cast<const uint4 *>(hb + (size_t)(start + src[u]) * pos_stride);
#pragma unroll
                for (int u = 0; u < KV_GROUP; ++u)
                    if (src[u] != j0 + u) *reinterpret_cast<uint4 *>(hb + (size_t)(start + j0 + u) * pos_stride) = val[u];
            }
        }
    }
    (void)bump;
}

__global__ void kv_bump_kernel(int32_t *cache_len, const int32_t *accept_len, int batch) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < batch) cache_len[b] += accept_len[b];
}

extern "C" int samd_kv_compact(void *const *kv_ptrs_dev, int32_t n_kv, int32_t n_heads, int32_t row_bytes, int64_t kv_batch_stride,
                               int64_t kv_head_stride, int64_t kv_pos_stride, const int32_t *indices_dev, int32_t depth,
                               const int32_t *accept_len_dev, int32_t *cache_len_dev, int32_t batch, void *stream) {
    SAMD_REQUIRE(accept_len_dev && cache_len_dev && batch > 0, "samd_kv_compact: bad arguments");
    if (indices_dev) {                                          // indices NULL = sequence draft: only the length bump
        SAMD_REQUIRE(kv_ptrs_dev && n_kv > 0 && n_heads > 0 && depth > 0, "samd_kv_compact: bad KV shape");
        SAMD_REQUIRE(row_bytes > 0 && row_bytes % 16 == 0 && kv_pos_stride % 16 == 0 && kv_head_stride % 16 == 0 &&
                         kv_batch_stride % 16 == 0,
                     "samd_kv_compact: KV rows must be 16-byte aligned");
        const int items = batch * n_kv;
        const int grid = std::min((items + VW - 1) / VW, 148 * 8);
        kv_compact_kernel<<<grid, VT, 0, (cudaStream_t)stream>>>(kv_ptrs_dev, n_kv, n_heads, row_bytes, kv_batch_stride,
                                                                 kv_head_stride, kv_pos_stride, indices_dev, depth, accept_len_dev,
                                                                 cache_len_dev, batch, 0);
        samd_count_launch();
        SAMD_CUDA(cudaGetLastError());
    }
    kv_bump_kernel<<<(batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(cache_len_dev, accept_len_dev, batch);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// Prefix rows from one KV cache into another (prefix reuse at admission): pair i copies rows [0, n_rows[i]) of batch row
// src_row[i] into batch row dst_row[i], every tensor and head.  blockIdx.y = pair; its rows are cut into 16-byte chunks
// (consecutive threads -> consecutive chunks of one row, so a head's rows stream contiguously) and every lane keeps
// CP_UNROLL chunks in flight.  A chunk whose two addresses are 16-byte aligned and that lies inside the row moves as one
// uint4; the row's partial last chunk, or any chunk of a row that is not 16-byte aligned, moves in the widest of 4 / 2 / 1
// bytes both addresses allow.
// ---------------------------------------------------------------------------------------
#define CP_THREADS 256
#define CP_UNROLL 4

struct KvSide {
    void *const *ptrs;
    long long batch_stride, head_stride, pos_stride;
};

__device__ __forceinline__ void copy_bytes(char *d, const char *s, int n) {
    const unsigned a = (unsigned)(((uintptr_t)d | (uintptr_t)s) & 3) | (unsigned)(n & 3);
    if (a == 0) {
        for (int k = 0; k < n; k += 4) *reinterpret_cast<uint32_t *>(d + k) = *reinterpret_cast<const uint32_t *>(s + k);
    } else if ((a & 1) == 0) {
        for (int k = 0; k < n; k += 2) *reinterpret_cast<uint16_t *>(d + k) = *reinterpret_cast<const uint16_t *>(s + k);
    } else {
        for (int k = 0; k < n; ++k) d[k] = s[k];
    }
}

__global__ void __launch_bounds__(CP_THREADS) kv_copy_rows_kernel(KvSide dst, KvSide src, int n_kv, int n_heads, int row_bytes,
                                                                  const int32_t *dst_row, const int32_t *src_row,
                                                                  const int32_t *n_rows) {
    const int p = blockIdx.y;
    const long long rows = n_rows[p];
    if (rows <= 0) return;
    const int cols = (row_bytes + 15) >> 4;
    const long long total = (long long)n_kv * n_heads * rows * cols;
    const long long db = (long long)dst_row[p] * dst.batch_stride, sb = (long long)src_row[p] * src.batch_stride;
    const long long stride = (long long)gridDim.x * CP_THREADS;
    for (long long u0 = (long long)blockIdx.x * CP_THREADS + threadIdx.x; u0 < total; u0 += stride * CP_UNROLL) {
        char *dp[CP_UNROLL];
        const char *sp[CP_UNROLL];
        int nb[CP_UNROLL];
        uint4 v[CP_UNROLL];
#pragma unroll
        for (int k = 0; k < CP_UNROLL; ++k) {
            const long long u = u0 + k * stride;
            nb[k] = 0;
            if (u >= total) continue;
            const int col = (int)(u % cols);
            long long rest = u / cols;
            const long long row = rest % rows;
            rest /= rows;
            const int hd = (int)(rest % n_heads), kv = (int)(rest / n_heads);
            const long long off = (long long)col << 4;
            dp[k] = reinterpret_cast<char *>(dst.ptrs[kv]) + db + hd * dst.head_stride + row * dst.pos_stride + off;
            sp[k] = reinterpret_cast<const char *>(src.ptrs[kv]) + sb + hd * src.head_stride + row * src.pos_stride + off;
            nb[k] = min(16, row_bytes - (int)off);
            if (nb[k] == 16 && (((uintptr_t)dp[k] | (uintptr_t)sp[k]) & 15) == 0) {
                v[k] = *reinterpret_cast<const uint4 *>(sp[k]);
                nb[k] = -16;                                             // vector chunk, loaded
            }
        }
#pragma unroll
        for (int k = 0; k < CP_UNROLL; ++k) {
            if (nb[k] == -16) *reinterpret_cast<uint4 *>(dp[k]) = v[k];
            else if (nb[k] > 0) copy_bytes(dp[k], sp[k], nb[k]);
        }
    }
}

extern "C" int samd_kv_copy_rows(void *const *dst_ptrs_dev, int64_t dst_batch_stride, int64_t dst_head_stride,
                                 int64_t dst_pos_stride, void *const *src_ptrs_dev, int64_t src_batch_stride,
                                 int64_t src_head_stride, int64_t src_pos_stride, int32_t n_kv, int32_t n_heads,
                                 int32_t row_bytes, const int32_t *dst_row_dev, const int32_t *src_row_dev,
                                 const int32_t *n_rows_dev, int32_t n_pairs, void *stream) {
    SAMD_REQUIRE(n_pairs >= 0 && n_pairs <= 65535, "samd_kv_copy_rows: n_pairs must be in [0, 65535]");
    if (n_pairs == 0) return 0;
    SAMD_REQUIRE(dst_ptrs_dev && src_ptrs_dev && dst_row_dev && src_row_dev && n_rows_dev,
                 "samd_kv_copy_rows: null pointer argument");
    SAMD_REQUIRE(n_kv > 0 && n_heads > 0 && row_bytes > 0, "samd_kv_copy_rows: bad KV shape");
    // about eight CTAs per SM in all, whatever the pair count: the grid depends on n_pairs only
    const unsigned per_pair = (unsigned)std::min(1024, std::max(8, (148 * 8 + n_pairs - 1) / n_pairs));
    const KvSide d{dst_ptrs_dev, dst_batch_stride, dst_head_stride, dst_pos_stride};
    const KvSide s{src_ptrs_dev, src_batch_stride, src_head_stride, src_pos_stride};
    kv_copy_rows_kernel<<<dim3(per_pair, (unsigned)n_pairs), CP_THREADS, 0, (cudaStream_t)stream>>>(
        d, s, n_kv, n_heads, row_bytes, dst_row_dev, src_row_dev, n_rows_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// TokenRecycle.gen_draft (samd/tree_model/token_recycle/token_recycle.py:49-59): one warp per request fills the
// static tree level by level from the [vocab][8] successor table (a node's token is known once its parent's is).
// ---------------------------------------------------------------------------------------
__global__ void recycle_tree_kernel(const int32_t *table, int vocab, const int32_t *parent, const int32_t *rank, int n_nodes,
                                    const int32_t *start_tok, const int32_t *type, int only_type, int batch, int32_t *out) {
    extern __shared__ int s_tree[];                            // [warps][2][n_nodes]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * (blockDim.x >> 5) + warp;
    if (b >= batch || (type && type[b] != only_type)) return;
    int *tok = s_tree + warp * 2 * n_nodes, *nxt = tok + n_nodes;
    constexpr int PENDING = INT_MIN;                            // (any real token id, even an invalid negative one, is final)
    for (int i = lane; i < n_nodes; i += 32) tok[i] = i == 0 ? max(start_tok[b], PENDING + 1) : PENDING;
    __syncwarp();
    // parents precede children, so each sweep settles at least one more level; depth <= n_nodes sweeps, 6 for the
    // reference's 61-node tree.  A sweep reads `tok` and writes `nxt`; the two are merged between sweeps.
    for (bool again = true; again;) {
        bool pending = false;
        for (int i = lane; i < n_nodes; i += 32) {
            int v = tok[i];
            if (v == PENDING) {
                const int pt = tok[parent[i]];
                if (pt == PENDING) {
                    pending = true;
                } else {
                    v = 0;                                      // no entry for the parent's token: stays 0
                    if (pt >= 0 && pt < vocab && rank[i] < TOPK && __ldg(table + (size_t)pt * TOPK) >= 0) v = __ldg(table + (size_t)pt * TOPK + rank[i]);
                }
            }
            nxt[i] = v;
        }
        __syncwarp();
        for (int i = lane; i < n_nodes; i += 32) tok[i] = nxt[i];
        __syncwarp();
        again = __any_sync(SAMD_FULL, pending);
    }
    for (int i = lane; i < n_nodes; i += 32) out[(size_t)b * n_nodes + i] = tok[i];
}

extern "C" int samd_recycle_gen_tree(const int32_t *table_dev, int32_t vocab, const int32_t *parent_dev, const int32_t *rank_dev,
                                     int32_t n_nodes, const int32_t *start_tok_dev, const int32_t *type_dev, int32_t only_type,
                                     int32_t batch, int32_t *out_tokens_dev, void *stream) {
    SAMD_REQUIRE(table_dev && parent_dev && rank_dev && start_tok_dev && out_tokens_dev, "samd_recycle_gen_tree: bad arguments");
    SAMD_REQUIRE(vocab > 0 && n_nodes > 0 && n_nodes <= 4096 && batch > 0, "samd_recycle_gen_tree: bad shape");
    const int warps = 4;
    recycle_tree_kernel<<<(batch + warps - 1) / warps, warps * 32, (size_t)warps * 2 * n_nodes * sizeof(int), (cudaStream_t)stream>>>(
        table_dev, vocab, parent_dev, rank_dev, n_nodes, start_tok_dev, type_dev, only_type, batch, out_tokens_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
