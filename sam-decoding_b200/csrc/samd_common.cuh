// Shared device/host definitions of the flat suffix-automaton layout (sm_100a).
//
// Layout (identical for the per-request dynamic arenas and the static automaton):
//   state record  16 x int32 = 64 B, 64-byte aligned (two sectors of one cache line):
//                   [0] link  [1] length  [2] min_endpos  [3] overflow list head (oldest)
//                   [4..8] inline edge tokens (SAMD_EMPTY = free)   [9..13] inline edge targets
//                   [14] overflow list tail (newest)   [15] aux
//                 The first five out-edges of a state live INSIDE its record, so a transition
//                 probe, the suffix link, the length and min_endpos all come from ONE 64-byte read,
//                 and clone-on-split is one 64-byte copy.  (Mean out-degree of non-root states is
//                 ~1.3; SURVEY.md section 8d.)
//   overflow edge uint4 {state, token, target, next (towards newer)} in an open-addressing table
//                 keyed (state, token): 8-slot (128 B) buckets, linear over buckets, a slot is free
//                 when .x == SAMD_EMPTY.  Nothing is ever deleted, so a probe ends at the first
//                 bucket that still has a free slot.  Per-state lists run oldest -> newest, so edge
//                 enumeration (clone, export, top-k) sees dict insertion order: inline, then the list.
//   text          int32, 1-based, text[0] = -1                         (dyn_sam.py:20)
// Tokens must be non-negative (SAMD_EMPTY = -1 marks free inline edges).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define SAMD_EMPTY 0xFFFFFFFFu
#define SAMD_NIL   0xFFFFFFFFu
#define SAMD_FULL  0xFFFFFFFFu
#define SAMD_BUCKET 8
#define SAMD_REC 16            // int32 words per state record
#define SAMD_INLINE 5          // inline out-edges per state

enum { R_LINK = 0, R_LEN = 1, R_END = 2, R_OHEAD = 3, R_TOK = 4, R_TGT = 9, R_OTAIL = 14, R_AUX = 15 };

enum { META_NSTATES = 0, META_LAST = 1, META_N = 2, META_CUR = 3, META_CURLEN = 4, META_NEDGES = 5,
       META_OVERFLOW = 6, META_NCLONES = 7, META_HOPS = 8, META_PROBES = 9, META_LASTLINK = 10,
       // when the newest append split a state: last_link is the clone, LLTWIN the state it copied (-1 = none), see sam_scalar.cuh
       META_LLTWIN = 11, META_LLLEN = 12, META_LLLINK = 13,
       META_MAXCHAIN = 14,    // longest cursor fallback chain any append of this request has seen (test / profiling counter)
       META_WORDS = 16 };

__host__ __device__ __forceinline__ uint32_t samd_hash(uint32_t state, uint32_t tok) {
    uint32_t h = state * 0x9E3779B1u + tok * 0x85EBCA77u;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 13;
    return h;
}

static inline uint64_t samd_next_pow2(uint64_t x) {
    uint64_t p = 1;
    while (p < x) p <<= 1;
    return p;
}
// overflow-table capacity rule for a growing automaton: >= 4 slots per token (edges <= 3n-4)
static inline uint64_t samd_table_slots(uint64_t n_tokens) {
    uint64_t c = samd_next_pow2(4 * (n_tokens + 1));
    return c < 64 ? 64 : c;
}

static inline void samd_init_rec(int32_t *w, int link, int len, int endpos) {
    w[R_LINK] = link;
    w[R_LEN] = len;
    w[R_END] = endpos;
    w[R_OHEAD] = (int32_t)SAMD_NIL;
    for (int i = 0; i < SAMD_INLINE; ++i) {
        w[R_TOK + i] = (int32_t)SAMD_EMPTY;
        w[R_TGT + i] = 0;
    }
    w[R_OTAIL] = (int32_t)SAMD_NIL;
    w[R_AUX] = 0;
}

struct DynArena {
    int32_t  *recs;     // [B][s_cap][SAMD_REC]
    uint4    *slots;    // [B][h_cap] overflow edges
    int32_t  *text;     // [B][t_cap]
    int32_t  *meta;     // [B][META_WORDS]
    int32_t   n_requests, max_tokens;
    uint32_t  s_cap, h_cap, t_cap, bmask;
};

struct StaticDev {
    const int32_t *recs;   // [n_states][SAMD_REC]
    const uint4   *slots;  // [n_slots] overflow edges
    const int32_t *text;
    const int32_t *occ;    // cnt_endpos (count flavour) or NULL
    const int2    *topk;   // [n_states][8] (token,target), -1 padded, or NULL
    int64_t  n_states, n_slots, n_tokens;
    uint32_t bmask;
};

struct samd_static_s {
    StaticDev dev;
    // host mirrors kept for export/save (test + persistence paths)
    int32_t  *h_recs;
    uint4    *h_slots;
    int32_t  *h_text;
    int32_t  *h_occ;
    int2     *h_topk;
    int64_t   n_edges, n_clones, n_ovf;
    int       with_counts;
    int       device;
};

struct samd_dyn_s {
    DynArena a;
    int32_t *tickets;   // [n_requests] arrival counters of samd_dyn_clone (0 between launches)
    int device;
    int64_t bytes;
};

void samd_set_error(const char *fmt, ...);
void samd_count_launch(int n = 1);

#define SAMD_CUDA(call)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            samd_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return 1;                                                                            \
        }                                                                                        \
    } while (0)

#define SAMD_REQUIRE(cond, msg)                                       \
    do {                                                              \
        if (!(cond)) {                                                \
            samd_set_error("%s (%s:%d)", msg, __FILE__, __LINE__);    \
            return 2;                                                 \
        }                                                             \
    } while (0)

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------
// Warp-cooperative transition probe.  Lanes 0..15 read the sixteen words of the state record (one
// 64 B request); the inline edges are matched with a ballot.  Only states with more than five
// out-edges (the root, a few hubs) ever touch the overflow table: lanes 0..7 then read one bucket.
// ---------------------------------------------------------------------------------------
struct Look {
    int      w;        // this lane's word of the record (valid in lanes 0..15)
    int      target;   // transition target when found
    uint32_t slot;     // overflow slot of the hit / first free overflow slot (when probed), else NIL
    int      k;        // inline index of the hit, or -1
    bool     found;
    bool     probed;   // the overflow table was searched (slot is meaningful)
};

__device__ __forceinline__ int rec_word(const Look &r, int which) { return __shfl_sync(SAMD_FULL, r.w, which); }

// a request's token count as the kernels use it: never negative, never beyond its row of the token block
__device__ __forceinline__ int samd_clamp_count(int c, int stride) { return min(max(c, 0), stride); }

// search the overflow table for (state, tok): found -> slot/target; else slot = first free slot
__device__ __forceinline__ void ovf_probe(const uint4 *slots, uint32_t bmask, uint32_t state, uint32_t tok, int lane,
                                          bool ro, Look &r) {
    uint32_t b = samd_hash(state, tok) & bmask;
    r.probed = true;
    while (true) {
        uint4 s = make_uint4(0xFFFFFFFEu, 0, 0, 0);
        if (lane < SAMD_BUCKET) {
            const uint4 *ptr = slots + ((size_t)b * SAMD_BUCKET + lane);
            s = ro ? __ldg(ptr) : *ptr;
        }
        const unsigned hit = __ballot_sync(SAMD_FULL, s.x == state && s.y == tok);
        const unsigned emp = __ballot_sync(SAMD_FULL, s.x == SAMD_EMPTY);
        if (hit) {
            const int l = __ffs(hit) - 1;
            r.found = true;
            r.slot = b * SAMD_BUCKET + l;
            r.target = (int)__shfl_sync(SAMD_FULL, s.z, l);
            return;
        }
        if (emp) {
            r.found = false;
            r.slot = b * SAMD_BUCKET + (__ffs(emp) - 1);
            return;
        }
        b = (b + 1) & bmask;
    }
}

// match `tok` against a record whose sixteen words are already held by lanes 0..15 (`w`)
template <bool kReadOnly>
__device__ __forceinline__ Look look_words(int w, const uint4 *slots, uint32_t bmask, int state, int tok, int lane) {
    Look r;
    r.w = w;
    r.slot = SAMD_NIL;
    r.probed = false;
    r.target = 0;
    const unsigned hit = __ballot_sync(SAMD_FULL, lane >= R_TOK && lane < R_TOK + SAMD_INLINE && w == tok);
    if (hit) {
        const int l = __ffs(hit) - 1;
        r.k = l - R_TOK;
        r.target = __shfl_sync(SAMD_FULL, w, l + (R_TGT - R_TOK));
        r.found = true;
        return r;
    }
    r.k = -1;
    r.found = false;
    if ((uint32_t)__shfl_sync(SAMD_FULL, w, R_OHEAD) != SAMD_NIL) ovf_probe(slots, bmask, (uint32_t)state, (uint32_t)tok, lane, kReadOnly, r);
    return r;
}

template <bool kReadOnly>
__device__ __forceinline__ Look warp_look(const int32_t *recs, const uint4 *slots, uint32_t bmask, int state, int tok, int lane) {
    const int32_t *p = recs + (size_t)state * SAMD_REC;
    int w = 0;
    if (lane < SAMD_REC) w = kReadOnly ? __ldg(p + lane) : p[lane];
    return look_words<kReadOnly>(w, slots, bmask, state, tok, lane);
}

// Hint: pull the 64 B record of `state` towards the SM (both sectors) ahead of its use.
__device__ __forceinline__ void prefetch_rec(const int32_t *recs, int state, int lane) {
    if (lane < 2) asm volatile("prefetch.global.L1 [%0];" ::"l"(recs + (size_t)state * SAMD_REC + lane * 8));
}

// Longest-suffix-match step (dyn_sam.py:69-78): one 64-byte read per suffix-link hop.
template <bool kReadOnly>
__device__ __forceinline__ void warp_transfer(const int32_t *recs, const uint4 *slots, uint32_t bmask, int &index, int &length,
                                              int tok, int lane, int &hops) {
    bool first = true;
    while (true) {
        const Look r = warp_look<kReadOnly>(recs, slots, bmask, index, tok, lane);
        hops++;
        if (!first) length = rec_word(r, R_LEN);        // length = states[index].length after a link hop
        if (r.found) {
            index = r.target;
            length += 1;
            return;
        }
        if (index == 0) {
            length = 0;
            return;
        }
        index = rec_word(r, R_LINK);
        if (index < 0) {                                 // only a scout racing with the builder can see a pending link
            index = 0;
            length = 0;
            return;
        }
        first = false;
    }
}
#endif  // __CUDACC__
