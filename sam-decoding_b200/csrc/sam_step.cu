// Dynamic-SAM arenas and the per-step draft kernel (extend + advance + lookup + select + draft).
// One CTA per request - a builder warp and up to three read-only scout warps that run ahead of it; see
// include/samd_b200.h for the reference methods each entry replaces.
#include "samd_common.cuh"
#include "sam_scalar.cuh"
#include "../../include/samd_b200.h"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

// ---------------------------------------------------------------------------------------
// arena management
// ---------------------------------------------------------------------------------------
__global__ void dyn_reset_kernel(DynArena a, const uint8_t *mask) {
    // one CTA per request: clear the overflow table (0xFF = free), fill EVERY record with the empty template {link -1,
    // length 0, min_endpos 0, no edges, no overflow list, aux 0} - which is also the root (dyn_sam.py:19) - so that
    // creating a state later only has to store its lengths (sam_scalar.cuh), and write the meta block
    int r = blockIdx.x;
    if (mask && !mask[r]) return;
    uint4 *slots = a.slots + (size_t)r * a.h_cap;
    const uint4 e = make_uint4(SAMD_EMPTY, SAMD_EMPTY, SAMD_EMPTY, SAMD_EMPTY);
    for (uint32_t i = threadIdx.x; i < a.h_cap; i += blockDim.x) slots[i] = e;
    int4 *recs4 = reinterpret_cast<int4 *>(a.recs + (size_t)r * a.s_cap * SAMD_REC);
    for (size_t i = threadIdx.x; i < (size_t)a.s_cap * 4; i += blockDim.x) {
        const int q = (int)(i & 3);          // words {-1,0,0,-1 | -1,-1,-1,-1 | -1,0,0,0 | 0,0,-1,0}
        recs4[i] = q == 0 ? make_int4(-1, 0, 0, -1) : q == 1 ? make_int4(-1, -1, -1, -1) : q == 2 ? make_int4(-1, 0, 0, 0) : make_int4(0, 0, -1, 0);
    }
    if (threadIdx.x == 0) {
        a.text[(size_t)r * a.t_cap] = -1;                                       // sentinel (dyn_sam.py:20)
        int32_t *m = a.meta + (size_t)r * META_WORDS;
        for (int i = 0; i < META_WORDS; ++i) m[i] = 0;
        m[META_NSTATES] = 1;
        m[META_LASTLINK] = -1;
        m[META_LLTWIN] = -1;
    }
}

extern "C" int samd_dyn_create(int n_requests, int max_tokens, samd_dyn_t *out) {
    SAMD_REQUIRE(n_requests > 0 && max_tokens > 0 && out, "samd_dyn_create: bad arguments");
    SAMD_REQUIRE(max_tokens < (1 << 28), "samd_dyn_create: max_tokens too large");
    samd_dyn_s *h = new samd_dyn_s();
    DynArena &a = h->a;
    a.n_requests = n_requests;
    a.max_tokens = max_tokens;
    a.s_cap = 2u * (uint32_t)max_tokens + 2u;                 // states <= 2n - 1 (+ root)
    a.h_cap = (uint32_t)samd_table_slots((uint64_t)max_tokens);
    a.t_cap = ((uint32_t)max_tokens + 1u + 3u) & ~3u;
    a.bmask = a.h_cap / SAMD_BUCKET - 1u;
    SAMD_CUDA(cudaGetDevice(&h->device));
    size_t b_recs = (size_t)n_requests * a.s_cap * SAMD_REC * sizeof(int32_t);
    size_t b_slots = (size_t)n_requests * a.h_cap * sizeof(uint4);
    size_t b_text = (size_t)n_requests * a.t_cap * sizeof(int32_t);
    size_t b_meta = (size_t)n_requests * META_WORDS * sizeof(int32_t);
    SAMD_CUDA(cudaMalloc(&a.recs, b_recs));
    SAMD_CUDA(cudaMalloc(&a.slots, b_slots));
    SAMD_CUDA(cudaMalloc(&a.text, b_text));
    SAMD_CUDA(cudaMalloc(&a.meta, b_meta));
    SAMD_CUDA(cudaMalloc(&h->tickets, (size_t)n_requests * sizeof(int32_t)));
    SAMD_CUDA(cudaMemset(h->tickets, 0, (size_t)n_requests * sizeof(int32_t)));
    h->bytes = (int64_t)(b_recs + b_slots + b_text + b_meta);
    *out = h;
    // the arenas are filled on the default stream; the caller's first launch may come on any other (non-blocking) stream
    // - torch's side streams do not order with the legacy default stream - so creation finishes the fill before returning
    if (int rc = samd_dyn_reset(h, nullptr, nullptr)) return rc;
    SAMD_CUDA(cudaDeviceSynchronize());
    return 0;
}

extern "C" int samd_dyn_destroy(samd_dyn_t h) {
    if (!h) return 0;
    cudaFree(h->a.recs);
    cudaFree(h->a.slots);
    cudaFree(h->a.text);
    cudaFree(h->a.meta);
    cudaFree(h->tickets);
    delete h;
    return 0;
}

extern "C" int64_t samd_dyn_bytes(samd_dyn_t h) { return h ? h->bytes : 0; }

extern "C" int samd_dyn_copy(samd_dyn_t dst, samd_dyn_t src, void *stream) {
    SAMD_REQUIRE(dst && src && dst->a.n_requests == src->a.n_requests && dst->a.max_tokens == src->a.max_tokens,
                 "samd_dyn_copy: handles must have the same shape");
    const DynArena &s = src->a;
    const DynArena &d = dst->a;
    cudaStream_t st = (cudaStream_t)stream;
    SAMD_CUDA(cudaMemcpyAsync(d.recs, s.recs, (size_t)s.n_requests * s.s_cap * SAMD_REC * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    SAMD_CUDA(cudaMemcpyAsync(d.slots, s.slots, (size_t)s.n_requests * s.h_cap * sizeof(uint4), cudaMemcpyDeviceToDevice, st));
    SAMD_CUDA(cudaMemcpyAsync(d.text, s.text, (size_t)s.n_requests * s.t_cap * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    SAMD_CUDA(cudaMemcpyAsync(d.meta, s.meta, (size_t)s.n_requests * META_WORDS * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return 0;
}

#define CLONE_THREADS 256
// One request of `s` onto one request of `d` (same s_cap / h_cap / t_cap): blockIdx.y = pair, gridDim.x CTAs share its
// 16-byte units - the live records [0, n_src), the EMPTY TEMPLATE over the destination's stale records [n_src, n_dst_old),
// the whole overflow table (hashed: no live prefix to follow) and text[0 .. max_length].  Every CTA reads n_dst_old from
// the destination's meta before it counts itself in on tickets[dst]; the last CTA to arrive - the others have all read it
// by then - writes the 16 meta words and clears the ticket for the next launch.
__global__ void __launch_bounds__(CLONE_THREADS) dyn_clone_kernel(DynArena d, const int32_t *dst_idx, DynArena s,
                                                                  const int32_t *src_idx, int32_t *tickets) {
    __shared__ int sh_old, sh_last;
    const int rd = dst_idx[blockIdx.y], rs = src_idx[blockIdx.y];
    if (rd < 0 || rd >= d.n_requests || rs < 0 || rs >= s.n_requests || (d.recs == s.recs && rd == rs)) return;
    const int32_t *sm = s.meta + (size_t)rs * META_WORDS;
    int32_t *dm = d.meta + (size_t)rd * META_WORDS;
    if (threadIdx.x == 0) {
        sh_old = dm[META_NSTATES];
        __threadfence();
        sh_last = atomicAdd(&tickets[rd], 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    const long long n_src = sm[META_NSTATES], n_old = sh_old;
    const long long u_rec = 4 * (n_src > n_old ? n_src : n_old);         // records: 4 units of 16 B each
    const long long u_tab = d.h_cap;
    const long long u_txt = ((long long)sm[META_N] + 1 + 3) >> 2;          // text[0 .. max_length], t_cap is a multiple of 4
    const int4 *srec = reinterpret_cast<const int4 *>(s.recs + (size_t)rs * s.s_cap * SAMD_REC);
    int4 *drec = reinterpret_cast<int4 *>(d.recs + (size_t)rd * d.s_cap * SAMD_REC);
    const uint4 *stab = s.slots + (size_t)rs * s.h_cap;
    uint4 *dtab = d.slots + (size_t)rd * d.h_cap;
    const int4 *stxt = reinterpret_cast<const int4 *>(s.text + (size_t)rs * s.t_cap);
    int4 *dtxt = reinterpret_cast<int4 *>(d.text + (size_t)rd * d.t_cap);
    const long long total = u_rec + u_tab + u_txt, stride = (long long)gridDim.x * CLONE_THREADS;
    for (long long u = (long long)blockIdx.x * CLONE_THREADS + threadIdx.x; u < total; u += stride) {
        if (u < u_rec) {
            if (u < 4 * n_src) {
                drec[u] = __ldg(srec + u);
            } else {                                                     // the template of dyn_reset_kernel
                const int q = (int)(u & 3);
                drec[u] = q == 0 ? make_int4(-1, 0, 0, -1) : q == 1 ? make_int4(-1, -1, -1, -1) : q == 2 ? make_int4(-1, 0, 0, 0) : make_int4(0, 0, -1, 0);
            }
        } else if (u < u_rec + u_tab) {
            dtab[u - u_rec] = __ldg(stab + (u - u_rec));
        } else {
            dtxt[u - u_rec - u_tab] = __ldg(stxt + (u - u_rec - u_tab));
        }
    }
    if (sh_last && threadIdx.x < META_WORDS) {
        dm[threadIdx.x] = sm[threadIdx.x];
        if (threadIdx.x == 0) tickets[rd] = 0;
    }
}

extern "C" int samd_dyn_clone(samd_dyn_t dst, const int32_t *dst_idx_dev, samd_dyn_t src, const int32_t *src_idx_dev,
                              int32_t n_pairs, void *stream) {
    SAMD_REQUIRE(dst && src && n_pairs >= 0, "samd_dyn_clone: bad arguments");
    if (dst->a.max_tokens != src->a.max_tokens) {
        samd_set_error("samd_dyn_clone: max_tokens differ (dst %d, src %d): the record, overflow-table and history "
                       "capacities must agree", dst->a.max_tokens, src->a.max_tokens);
        return 2;
    }
    if (n_pairs == 0) return 0;
    SAMD_REQUIRE(dst_idx_dev && src_idx_dev, "samd_dyn_clone: null index array");
    SAMD_REQUIRE(n_pairs <= 65535, "samd_dyn_clone: at most 65535 pairs per launch");
    // CTAs per pair from the capacity alone (about 16 units per thread at a full arena): no argument depends on the step
    const long long units = 4LL * dst->a.s_cap + dst->a.h_cap;
    const unsigned per_pair = (unsigned)std::max(4LL, std::min(64LL, units / (CLONE_THREADS * 16)));
    dyn_clone_kernel<<<dim3(per_pair, (unsigned)n_pairs), CLONE_THREADS, 0, (cudaStream_t)stream>>>(
        dst->a, dst_idx_dev, src->a, src_idx_dev, dst->tickets);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int samd_dyn_stats(samd_dyn_t h, int64_t *out) {
    // out[8] = sums over requests of {n_states, max_length, n_edges, n_clones, extend probes, lookup probes,
    //          requests whose arena overflowed, requests that were handed a negative token}
    SAMD_REQUIRE(h && out, "samd_dyn_stats: bad arguments");
    SAMD_CUDA(cudaDeviceSynchronize());
    const size_t n = (size_t)h->a.n_requests * META_WORDS;
    int32_t *m = (int32_t *)malloc(n * sizeof(int32_t));
    SAMD_CUDA(cudaMemcpy(m, h->a.meta, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 8; ++i) out[i] = 0;
    for (int r = 0; r < h->a.n_requests; ++r) {
        const int32_t *q = m + (size_t)r * META_WORDS;
        out[0] += q[META_NSTATES];
        out[1] += q[META_N];
        out[2] += q[META_NEDGES];
        out[3] += q[META_NCLONES];
        out[4] += q[META_HOPS];
        out[5] += q[META_PROBES];
        out[6] += q[META_OVERFLOW] & 1;
        out[7] += (q[META_OVERFLOW] >> 1) & 1;
    }
    free(m);
    return 0;
}

extern "C" int samd_dyn_meta(samd_dyn_t h, int32_t *meta_host) {
    SAMD_REQUIRE(h && meta_host, "samd_dyn_meta: bad arguments");
    SAMD_CUDA(cudaDeviceSynchronize());
    SAMD_CUDA(cudaMemcpy(meta_host, h->a.meta, (size_t)h->a.n_requests * META_WORDS * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" int samd_dyn_reset(samd_dyn_t h, const uint8_t *mask_dev, void *stream) {
    SAMD_REQUIRE(h, "samd_dyn_reset: null handle");
    dyn_reset_kernel<<<h->a.n_requests, 256, 0, (cudaStream_t)stream>>>(h->a, mask_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int samd_dyn_export(samd_dyn_t h, int request, int32_t *meta_host, int32_t *link_host, int32_t *length_host,
                               int32_t *endpos_host, int32_t *text_host, int64_t capacity) {
    SAMD_REQUIRE(h && request >= 0 && request < h->a.n_requests, "samd_dyn_export: bad request index");
    SAMD_CUDA(cudaDeviceSynchronize());
    int32_t meta[META_WORDS];
    SAMD_CUDA(cudaMemcpy(meta, h->a.meta + (size_t)request * META_WORDS, sizeof(meta), cudaMemcpyDeviceToHost));
    if (meta_host)
        for (int i = 0; i < 8; ++i) meta_host[i] = meta[i];
    int ns = meta[META_NSTATES];
    if (link_host || length_host || endpos_host) {
        SAMD_REQUIRE(capacity >= ns, "samd_dyn_export: capacity too small");
        int32_t *tmp = (int32_t *)malloc((size_t)ns * SAMD_REC * sizeof(int32_t));
        SAMD_CUDA(cudaMemcpy(tmp, h->a.recs + (size_t)request * h->a.s_cap * SAMD_REC, (size_t)ns * SAMD_REC * sizeof(int32_t),
                             cudaMemcpyDeviceToHost));
        for (int i = 0; i < ns; ++i) {
            if (link_host) link_host[i] = tmp[(size_t)i * SAMD_REC + R_LINK];
            if (length_host) length_host[i] = tmp[(size_t)i * SAMD_REC + R_LEN];
            if (endpos_host) endpos_host[i] = tmp[(size_t)i * SAMD_REC + R_END];
        }
        free(tmp);
    }
    if (text_host) {
        SAMD_REQUIRE(capacity >= meta[META_N] + 1, "samd_dyn_export: capacity too small for text");
        SAMD_CUDA(cudaMemcpy(text_host, h->a.text + (size_t)request * h->a.t_cap,
                             (size_t)(meta[META_N] + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost));
    }
    return 0;
}

// ---------------------------------------------------------------------------------------
// online append with clone-on-split (dyn_sam.py:41-67); registers are warp-uniform
// ---------------------------------------------------------------------------------------
struct DynRegs {
    int n_states, last, last_link, n, cur, cur_len, n_edges, n_clones, hops, max_chain;
};

// add the out-edge state --tok--> target, given the (failed) look-up `r` of (state, tok)
__device__ __forceinline__ void add_edge(int32_t *recs, uint4 *slots, uint32_t bmask, int state, int tok, int target, Look &r,
                                         int lane) {
    int32_t *rec = recs + (size_t)state * SAMD_REC;
    const unsigned emp = __ballot_sync(SAMD_FULL, lane >= R_TOK && lane < R_TOK + SAMD_INLINE && (uint32_t)r.w == SAMD_EMPTY);
    if (emp) {                                              // a free inline edge: two 4-byte stores
        const int l = __ffs(emp) - 1;
        if (lane == 0) {
            rec[l] = tok;
            rec[l + (R_TGT - R_TOK)] = target;
            rec[R_AUX] = l - R_TOK + 1;                     // inline-edge count (arena invariant, sam_scalar.cuh)
        }
        return;
    }
    if (!r.probed) ovf_probe(slots, bmask, (uint32_t)state, (uint32_t)tok, lane, false, r);
    const uint32_t tail = (uint32_t)rec_word(r, R_OTAIL);
    if (lane == 0) {
        slots[r.slot] = make_uint4((uint32_t)state, (uint32_t)tok, (uint32_t)target, SAMD_NIL);
        if (tail != SAMD_NIL) slots[tail].w = r.slot;     // append: lists run oldest -> newest
        else rec[R_OHEAD] = (int)r.slot;
        rec[R_OTAIL] = (int)r.slot;
    }
}

// ---------------------------------------------------------------------------------------
// The cursor's fallback chain for a token (transfer_cur_state: follow suffix links until a state has an edge on the
// token) visits exactly the states the append then gives that edge to (add_state walks the tail's suffix chain, and
// the cursor IS link(tail), up to the pre-clone quirk: then the chain is one stop longer at the front).  The
// transfer therefore leaves the chain in shared memory and the append inserts the edge at all of its stops at
// once, one lane per state, instead of walking it a second time, one dependent stop after the other.
// ---------------------------------------------------------------------------------------
#define CHAIN_MAX 64

// transfer_cur_state that records the states it visits (same walk as warp_transfer<false>); stopped_on_edge tells
// whether the last recorded state has the edge (else the walk ended at the root without finding one)
__device__ __forceinline__ void warp_transfer_chain(const int32_t *recs, const uint4 *slots, uint32_t bmask, int &index, int &length,
                                                    int tok, int lane, int &hops, int *chain, int &n_chain, bool &stopped_on_edge) {
    bool first = true;
    n_chain = 0;
    stopped_on_edge = false;
    while (true) {
        const Look r = warp_look<false>(recs, slots, bmask, index, tok, lane);
        if (lane == 0 && n_chain < CHAIN_MAX) chain[n_chain] = index;
        ++n_chain;                                           // > CHAIN_MAX: too long to replay, the append walks it itself
        hops++;
        if (!first) length = rec_word(r, R_LEN);
        if (r.found) {
            index = r.target;
            length += 1;
            stopped_on_edge = true;
            break;
        }
        if (index == 0) {
            length = 0;
            break;
        }
        index = rec_word(r, R_LINK);
        first = false;
    }
    __syncwarp();
}

// one lane, one state: give `state` the out-edge tok -> target (it has none on tok yet); the overflow slot is claimed
// with a compare-and-swap because two lanes of the same append may hash into the same bucket
__device__ __forceinline__ void lane_add_edge(int32_t *recs, uint4 *slots, uint32_t bmask, int state, int tok, int target) {
    int32_t *rec = recs + (size_t)state * SAMD_REC;
#pragma unroll
    for (int i = 0; i < SAMD_INLINE; ++i) {
        if ((uint32_t)rec[R_TOK + i] == SAMD_EMPTY) {
            rec[R_TOK + i] = tok;
            rec[R_TGT + i] = target;
            rec[R_AUX] = i + 1;
            return;
        }
    }
    uint32_t b = samd_hash((uint32_t)state, (uint32_t)tok) & bmask;
    while (true) {
        for (int l = 0; l < SAMD_BUCKET; ++l) {
            const uint32_t slot = b * SAMD_BUCKET + l;
            uint32_t *sx = reinterpret_cast<uint32_t *>(slots + slot);
            if (*reinterpret_cast<volatile uint32_t *>(sx) != SAMD_EMPTY) continue;
            if (atomicCAS(sx, SAMD_EMPTY, (uint32_t)state) != SAMD_EMPTY) continue;
            sx[1] = (uint32_t)tok;
            sx[2] = (uint32_t)target;
            sx[3] = SAMD_NIL;
            const uint32_t tail = (uint32_t)rec[R_OTAIL];
            if (tail != SAMD_NIL) slots[tail].w = slot;     // lists run oldest -> newest
            else rec[R_OHEAD] = (int)slot;
            rec[R_OTAIL] = (int)slot;
            return;
        }
        b = (b + 1) & bmask;
    }
}

template <bool kProf>                                       // kProf: the profiling build of the kernel (cycles by part in acc)
__device__ __forceinline__ void dyn_append(int32_t *recs, uint4 *slots, int32_t *text, uint32_t bmask, DynRegs &g, int tok,
                                           int lane, long long *acc, const int *chain, int n_chain, bool chain_on_edge) {
    g.n += 1;
    const int cur = g.n_states++;
    if (lane < SAMD_REC) {                                  // the new state's record: one 64-byte store
        int v = 0;
        if (lane == R_LINK || lane == R_OHEAD || lane == R_OTAIL || (lane >= R_TOK && lane < R_TOK + SAMD_INLINE)) v = -1;
        if (lane == R_LEN || lane == R_END) v = g.n;
        recs[(size_t)cur * SAMD_REC + lane] = v;
    }
    if (lane == 0) text[g.n] = tok;
    int p = g.last;
    int link_cur = 0;
    if (p != 0) {
        // `last` was created by the previous append and has no out-edge yet (edges are only ever added
        // along the suffix chain of the tail): write its first inline edge without reading anything.
        if (lane == 0) {
            recs[(size_t)p * SAMD_REC + R_TOK] = tok;
            recs[(size_t)p * SAMD_REC + R_TGT] = cur;
            recs[(size_t)p * SAMD_REC + R_AUX] = 1;
        }
        g.n_edges++;
        p = g.last_link;
    }
    __syncwarp();
    // the cursor's walk for this token already enumerated the stops that lack the edge: insert at all of them at once
    if (n_chain > 0 && n_chain <= CHAIN_MAX) {
        int s0 = -1;
        if (chain[0] == p) s0 = 0;
        else if (n_chain > 1 && chain[1] == p) s0 = 1;
        if (s0 >= 0) {
            const long long t0 = kProf ? clock64() : 0;
            const int end = chain_on_edge ? n_chain - 1 : n_chain;           // [s0, end): states without the edge
            for (int j = s0 + lane; j < end; j += 32) lane_add_edge(recs, slots, bmask, chain[j], tok, cur);
            g.n_edges += end - s0;
            __syncwarp();
            p = chain_on_edge ? chain[n_chain - 1] : -1;                     // resume at the state that has the edge
            if constexpr (kProf) acc[1] += clock64() - t0;
        }
    }
    while (p != -1) {
        long long t0 = kProf ? clock64() : 0;
        Look r = warp_look<false>(recs, slots, bmask, p, tok, lane);
        if constexpr (kProf) {
            const long long t = clock64();
            acc[0] += t - t0;                               // the chain's look-ups
            t0 = t;
        }
        if (!r.found) {
            add_edge(recs, slots, bmask, p, tok, cur, r, lane);
            if constexpr (kProf) acc[1] += clock64() - t0;              // edge inserts
            g.n_edges++;
            __syncwarp();
            p = rec_word(r, R_LINK);
            continue;
        }
        const int q = r.target;
        const long long tq0 = kProf ? clock64() : 0;
        // one request, two records: q's (lanes 0..15) and, speculatively, link(p)'s (lanes 16..31) - the
        // first state the redirect walk of a clone-on-split visits - so both DRAM reads overlap
        const int lp = rec_word(r, R_LINK);
        int qw = 0;
        if (lane < SAMD_REC) qw = recs[(size_t)q * SAMD_REC + lane];
        else if (lp >= 0) qw = recs[(size_t)lp * SAMD_REC + (lane - SAMD_REC)];
        const int lpw = __shfl_sync(SAMD_FULL, qw, (lane + SAMD_REC) & 31);      // link(p)'s words in lanes 0..15
        const int len_p = rec_word(r, R_LEN);
        const int len_q = __shfl_sync(SAMD_FULL, qw, R_LEN);
        if constexpr (kProf) acc[2] += clock64() - tq0;                 // the target's record (a dependent read)
        if (len_p + 1 == len_q) {
            link_cur = q;
        } else {
            // clone-on-split: the clone is q's record (inline edges, link, min_endpos) with length
            // len(p)+1 - one 64-byte copy; q's overflow edges, if any, are re-inserted oldest first
            const int clone = g.n_states++;
            g.n_clones++;
            int cw = qw;
            if (lane >= SAMD_REC) cw = 0;
            if (lane == R_LEN) cw = len_p + 1;
            if (lane == R_OHEAD || lane == R_OTAIL) cw = -1;
            if (lane < SAMD_REC) recs[(size_t)clone * SAMD_REC + lane] = cw;
            g.n_edges += __popc(__ballot_sync(SAMD_FULL, lane >= R_TOK && lane < R_TOK + SAMD_INLINE && (uint32_t)qw != SAMD_EMPTY));
            uint32_t e = (uint32_t)__shfl_sync(SAMD_FULL, qw, R_OHEAD);
            uint32_t head_c = SAMD_NIL, tail_c = SAMD_NIL;
            const long long tc0 = kProf ? clock64() : 0;
            while (e != SAMD_NIL) {
                const uint4 se = slots[e];
                if (lane == 0 && se.w != SAMD_NIL) asm volatile("prefetch.global.L1 [%0];" ::"l"(slots + se.w));
                Look f;
                f.found = false;
                ovf_probe(slots, bmask, (uint32_t)clone, se.y, lane, false, f);
                if (lane == 0) {
                    slots[f.slot] = make_uint4((uint32_t)clone, se.y, se.z, SAMD_NIL);
                    if (tail_c != SAMD_NIL) slots[tail_c].w = f.slot;
                }
                if (head_c == SAMD_NIL) head_c = f.slot;
                tail_c = f.slot;
                g.n_edges++;
                __syncwarp();
                e = se.w;
            }
            if (lane == 0 && head_c != SAMD_NIL) {
                recs[(size_t)clone * SAMD_REC + R_OHEAD] = (int)head_c;
                recs[(size_t)clone * SAMD_REC + R_OTAIL] = (int)tail_c;
            }
            const long long tc1 = kProf ? clock64() : 0;
            if constexpr (kProf) acc[3] += tc1 - tc0;                   // copy of q's overflow edges
            // redirect p's suffix chain from q to the clone
            Look cp = r;
            int pp = p;
            bool first_hop = true;
            while (true) {
                if (lane == 0) {
                    if (cp.k >= 0) recs[(size_t)pp * SAMD_REC + R_TGT + cp.k] = clone;
                    else slots[cp.slot].z = (uint32_t)clone;
                }
                __syncwarp();
                pp = rec_word(cp, R_LINK);
                if (pp == -1) break;
                // the first hop's record was fetched together with q's (nothing wrote to it since)
                cp = first_hop ? look_words<false>(lpw, slots, bmask, pp, tok, lane)
                               : warp_look<false>(recs, slots, bmask, pp, tok, lane);
                first_hop = false;
                if (!(cp.found && cp.target == q)) break;
            }
            if (lane == 0) recs[(size_t)q * SAMD_REC + R_LINK] = clone;
            link_cur = clone;
            if constexpr (kProf) acc[4] += clock64() - tc1;             // redirect walk
        }
        break;
    }
    if (lane == 0) recs[(size_t)cur * SAMD_REC + R_LINK] = link_cur;
    __syncwarp();
    g.last = cur;
    g.last_link = link_cur;
}

struct StepParams {
    DynArena dyn;
    StaticDev st;
    int has_static;
    int32_t *static_cursor;
    const int32_t *tokens;
    int token_stride;
    const int32_t *counts;
    const int32_t *start_tok;
    int flavour, n_predicts, len_bias, len_threshold;
    double alpha;
    int32_t *out_type, *out_match_dyn, *out_match_static, *out_index_dyn, *out_index_static, *out_draft, *out_draft_len;
    int draft_stride;
    long long *dbg_cycles;      // optional [10][n_requests] per-request SM cycles by phase (profiling hook, see samd_b200.h)
    int ngram;                  // depth of the short-context scouts (-1 = off)
    int prewalk;                // draft tokens the cursor scouts walk ahead for the next step (0 = off)
    int32_t *trace;             // optional [n_requests][trace_cap]: word 0 = count, then the states whose records the builder read
    int trace_cap;
};

#define SCOUT_MAX_TOKENS 64
// Scout warp: walks the cursor chain of the tokens this step will append (and of the final lookup) on the
// automaton AS IT IS - transfers only, nothing is written - one dependent read per token, i.e. faster than the
// builder warp, whose chain also carries clone / redirect work.  Every record (and the draft's text lines) it
// touches lands in this SM's L1/L2 just before the builder needs it.  It may observe records the builder is
// updating concurrently; that can only send it down a different (still valid) path - it is a prefetcher and
// produces no output.
template <bool kStatic>
__device__ __forceinline__ void scout_walk(const int32_t *recs, const uint4 *slots, uint32_t bmask, const int32_t *text,
                                           int idx, const int32_t *tk, int k, int peek, int n_predicts, long long text_n,
                                           long long cap, int lane, int *mailbox = nullptr) {
    // `cap` bounds every state index before it is dereferenced: the scout races with the builder and may read a
    // record whose initialisation is not visible yet (stale memory), so nothing it reads is trusted as an address
    if (k > SCOUT_MAX_TOKENS) return;                                        // long appends (prefill): nothing useful to scout
    if ((unsigned long long)idx >= (unsigned long long)cap) return;
    const int total = k + (peek >= 0 ? 1 : 0);
    int mine = 0;
    for (int i = 0; i < total; ++i) {
        if ((i & 31) == 0) mine = (i + lane < k) ? tk[i + lane] : peek;      // tokens, then the lookup token
        const int tok = __shfl_sync(SAMD_FULL, mine, i & 31);
        int up_state = 0, up_target = 0;                                     // for the redirect scout
        while (true) {                                                       // transfer_state, no bookkeeping
            const Look r = warp_look<kStatic>(recs, slots, bmask, idx, tok, lane);
            if (r.found) {
                if (!kStatic && i < k) {
                    // the builder reads the target's record together with the record of the stop above this one (the
                    // first stop of a clone's redirect walk): request that one too, without waiting for it
                    const int up = rec_word(r, R_LINK);
                    if (up > 0 && (unsigned long long)up < (unsigned long long)cap) prefetch_rec(recs, up, lane);
                    up_state = up;
                    up_target = r.target;
                }
                idx = r.target;
                if ((unsigned long long)idx >= (unsigned long long)cap) idx = 0;
                break;
            }
            if (idx == 0) break;
            idx = rec_word(r, R_LINK);
            if ((unsigned long long)idx >= (unsigned long long)cap) {
                idx = 0;
                break;
            }
        }
        if (!kStatic && mailbox && i < k && lane == 0) {     // every token gets an entry (stop 0 = nothing to look up)
            atomicExch(&mailbox[4 * i + 0], up_state);       // (atomics: a defined hand-off between two warps of the CTA)
            atomicExch(&mailbox[4 * i + 1], tok);
            atomicExch(&mailbox[4 * i + 2], up_target);
            __threadfence_block();
            atomicExch(&mailbox[4 * SCOUT_MAX_TOKENS], i + 1);
        }
    }
    if (peek < 0) return;
    // the draft will be read right after the earliest end position of the matched state
    const int e = kStatic ? __ldg(recs + (size_t)idx * SAMD_REC + R_END) : recs[(size_t)idx * SAMD_REC + R_END];
    if (e >= 0 && lane * 8 < n_predicts + 8 && (long long)e + 1 + lane * 8 <= text_n)
        asm volatile("prefetch.global.L1 [%0];" ::"l"(text + e + 1 + lane * 8));
}

// Redirect scout.  When the builder has to split the state an edge leads to (clone-on-split, 0.7 times per token on
// copy-heavy streams) it re-points that edge at the states further up the suffix chain - a cold pointer chase that
// neither the cursor's walk nor the first scout has touched.  This warp takes (stop above, token, target) hand-offs
// from the first scout and looks the next few stops up, so that their records and buckets are in cache.
__device__ __forceinline__ void redirect_scout(const int32_t *recs, const uint4 *slots, uint32_t bmask, int *mailbox,
                                               int k, long long cap, int lane) {
    if (k > SCOUT_MAX_TOKENS) return;
    for (int i = 0; i < k; ++i) {
        int have = 0;
        if (lane == 0) {
            while (true) {
                if (atomicAdd(&mailbox[4 * SCOUT_MAX_TOKENS], 0) > i) {
                    have = 1;
                    break;
                }
                if (atomicAdd(&mailbox[4 * SCOUT_MAX_TOKENS + 1], 0)) break;   // the first scout is done and never got this far
                __nanosleep(40);
            }
        }
        have = __shfl_sync(SAMD_FULL, have, 0);
        if (!have) return;
        __threadfence_block();
        int pp = 0, tok = 0, target = 0;
        if (lane == 0) {
            pp = atomicAdd(&mailbox[4 * i + 0], 0);
            tok = atomicAdd(&mailbox[4 * i + 1], 0);
            target = atomicAdd(&mailbox[4 * i + 2], 0);
        }
        pp = __shfl_sync(SAMD_FULL, pp, 0);
        tok = __shfl_sync(SAMD_FULL, tok, 0);
        target = __shfl_sync(SAMD_FULL, target, 0);
        for (int up = 0; up < 6 && pp > 0 && (unsigned long long)pp < (unsigned long long)cap; ++up) {
            const Look ru = warp_look<false>(recs, slots, bmask, pp, tok, lane);
            if (!ru.found || ru.target != target) break;
            pp = rec_word(ru, R_LINK);
        }
    }
}

template <bool kProf>
__global__ void __launch_bounds__(128) sam_step_kernel(StepParams P) {
    __shared__ int s_mailbox[4 * SCOUT_MAX_TOKENS + 2];        // first scout -> redirect scout
    const int r = blockIdx.x;
    const int lane = threadIdx.x & 31;
    if (r >= P.dyn.n_requests) return;
    if (threadIdx.x < 2) s_mailbox[4 * SCOUT_MAX_TOKENS + threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x >= 32) {
        const int k = P.tokens ? (P.counts ? samd_clamp_count(P.counts[r], P.token_stride) : P.token_stride) : 0;
        const int32_t *tk = P.tokens ? P.tokens + (size_t)r * P.token_stride : nullptr;
        const int peek = P.start_tok ? P.start_tok[r] : -1;
        if (threadIdx.x < 64) {
            const int32_t *meta = P.dyn.meta + (size_t)r * META_WORDS;
            scout_walk<false>(P.dyn.recs + (size_t)r * P.dyn.s_cap * SAMD_REC, P.dyn.slots + (size_t)r * P.dyn.h_cap, P.dyn.bmask,
                              P.dyn.text + (size_t)r * P.dyn.t_cap, meta[META_CUR], tk, k, peek, P.n_predicts, (long long)meta[META_N],
                              (long long)P.dyn.s_cap, lane, blockDim.x > 96 ? s_mailbox : nullptr);
            if (lane == 0) {                                  // whatever path the scout left by: no more hand-offs
                __threadfence_block();
                atomicExch(&s_mailbox[4 * SCOUT_MAX_TOKENS + 1], 1);
            }
        } else if (threadIdx.x >= 96) {
            redirect_scout(P.dyn.recs + (size_t)r * P.dyn.s_cap * SAMD_REC, P.dyn.slots + (size_t)r * P.dyn.h_cap, P.dyn.bmask, s_mailbox,
                           k, (long long)P.dyn.s_cap, lane);
        } else if (P.has_static) {
            scout_walk<true>(P.st.recs, P.st.slots, P.st.bmask, P.st.text, P.static_cursor[2 * r], tk, k, peek, P.n_predicts,
                             (long long)P.st.n_tokens, (long long)P.st.n_states, lane);
        }
        return;
    }
    __shared__ int s_chain[CHAIN_MAX];
    int n_chain = 0;
    bool chain_on_edge = false;
    const long long t_begin = kProf ? clock64() : 0;
    long long c_transfer = 0, c_append = 0, t_mark = 0;
    long long acc[5] = {0, 0, 0, 0, 0};
    int32_t *recs = P.dyn.recs + (size_t)r * P.dyn.s_cap * SAMD_REC;
    uint4 *slots = P.dyn.slots + (size_t)r * P.dyn.h_cap;
    int32_t *text = P.dyn.text + (size_t)r * P.dyn.t_cap;
    int32_t *meta = P.dyn.meta + (size_t)r * META_WORDS;
    const uint32_t bmask = P.dyn.bmask;

    DynRegs g;
    {
        int m = (lane < META_WORDS) ? meta[lane] : 0;
        g.n_states = __shfl_sync(SAMD_FULL, m, META_NSTATES);
        g.last = __shfl_sync(SAMD_FULL, m, META_LAST);
        g.last_link = __shfl_sync(SAMD_FULL, m, META_LASTLINK);
        g.n = __shfl_sync(SAMD_FULL, m, META_N);
        g.cur = __shfl_sync(SAMD_FULL, m, META_CUR);
        g.cur_len = __shfl_sync(SAMD_FULL, m, META_CURLEN);
        g.n_edges = __shfl_sync(SAMD_FULL, m, META_NEDGES);
        g.n_clones = __shfl_sync(SAMD_FULL, m, META_NCLONES);
        g.hops = __shfl_sync(SAMD_FULL, m, META_HOPS);
        g.max_chain = __shfl_sync(SAMD_FULL, m, META_MAXCHAIN);
    }
    int s_idx = 0, s_len = 0, s_hops = 0;
    if (P.has_static) {
        s_idx = P.static_cursor[2 * r];
        s_len = P.static_cursor[2 * r + 1];
    }

    // ---- phase 1: DraftModel.update (draft.py:65-79) ------------------------------------
    if (P.tokens) {
        const int k = P.counts ? samd_clamp_count(P.counts[r], P.token_stride) : P.token_stride;
        const int32_t *tk = P.tokens + (size_t)r * P.token_stride;
        bool overflow = false;
        prefetch_rec(recs, g.cur, lane);
        if (P.has_static) prefetch_rec(P.st.recs, s_idx, lane);
        for (int i = 0; i < k; i += 32) {
            const int mine = (i + lane < k) ? tk[i + lane] : 0;     // coalesced token fetch
            const int lim = min(32, k - i);
            for (int j = 0; j < lim; ++j) {
                const int tok = __shfl_sync(SAMD_FULL, mine, j);
                if (g.n >= P.dyn.max_tokens) {
                    overflow = true;
                    break;
                }
                // add_tokens: match first, then append (dyn_sam.py:84-88); StaticSAM.transfer_tokens
                // (static_sam.py:102-104) walks an independent structure, so it goes first too
                if constexpr (kProf) t_mark = clock64();
                warp_transfer_chain(recs, slots, bmask, g.cur, g.cur_len, tok, lane, g.hops, s_chain, n_chain, chain_on_edge);
                g.max_chain = max(g.max_chain, n_chain);
                if (P.has_static) warp_transfer<true>(P.st.recs, P.st.slots, P.st.bmask, s_idx, s_len, tok, lane, s_hops);
                if constexpr (kProf) {
                    const long long t = clock64();
                    c_transfer += t - t_mark;
                    t_mark = t;
                }
                // the records the NEXT token (or the final lookup) starts from are known now
                prefetch_rec(recs, g.cur, lane);
                if (P.has_static) prefetch_rec(P.st.recs, s_idx, lane);
                dyn_append<kProf>(recs, slots, text, bmask, g, tok, lane, acc, s_chain, n_chain, chain_on_edge);
                if constexpr (kProf) c_append += clock64() - t_mark;
            }
            if (overflow) break;
        }
        if (lane == 0) {
            meta[META_NSTATES] = g.n_states;
            meta[META_LAST] = g.last;
            meta[META_LASTLINK] = g.last_link;
            meta[META_N] = g.n;
            meta[META_CUR] = g.cur;
            meta[META_CURLEN] = g.cur_len;
            meta[META_NEDGES] = g.n_edges;
            meta[META_NCLONES] = g.n_clones;
            meta[META_HOPS] = g.hops;
            meta[META_LLTWIN] = -1;                  // (the one-thread kernel's hint; this kernel does not keep it)
            meta[META_MAXCHAIN] = g.max_chain;
            if (overflow) meta[META_OVERFLOW] = 1;
            if (P.has_static) {
                P.static_cursor[2 * r] = s_idx;
                P.static_cursor[2 * r + 1] = s_len;
            }
        }
    }
    if (!P.start_tok) return;
    const long long t_lookup = kProf ? clock64() : 0;

    // ---- phase 2: DraftModel.lookup (draft.py:52-63 / samd_sam_only/draft.py:49-59) -------
    const int tok = P.start_tok[r];
    int d_idx = g.cur, d_len = g.cur_len;
    int q_hops = 0;
    warp_transfer<false>(recs, slots, bmask, d_idx, d_len, tok, lane, q_hops);
    int t_idx = 0, t_len = 0;
    if (P.has_static) {
        t_idx = s_idx;
        t_len = s_len;
        warp_transfer<true>(P.st.recs, P.st.slots, P.st.bmask, t_idx, t_len, tok, lane, s_hops);
    }
    const int t_biased = t_len - P.len_bias;
    int type, n_out, endpos = 0, text_n = 0;
    const int32_t *src = nullptr;
    if (P.flavour == SAMD_FLAVOUR_SAMD) {
        n_out = P.n_predicts;
        if (max(d_len, t_biased) >= P.len_threshold) {
            if (d_len >= t_biased) {
                type = SAMD_DRAFT_DYN_SEQ;
                // to_anc (dyn_sam.py:99-105)
                int idx = d_idx;
                int4 rec = *reinterpret_cast<const int4 *>(recs + (size_t)idx * SAMD_REC);
                if (idx != 0) {
                    while (rec.x != 0 && P.n_predicts > g.n - rec.z) {
                        idx = rec.x;
                        rec = *reinterpret_cast<const int4 *>(recs + (size_t)idx * SAMD_REC);
                    }
                }
                endpos = rec.z;
                src = text;
                text_n = g.n;
            } else {
                type = SAMD_DRAFT_STATIC_SEQ;
                endpos = __ldg(P.st.recs + (size_t)t_idx * SAMD_REC + R_END);
                src = P.st.text;
                text_n = (int)P.st.n_tokens;
            }
        } else {
            type = SAMD_DRAFT_TREE_MODEL;
            n_out = 0;
        }
    } else {
        if (d_len >= t_biased) {
            type = SAMD_DRAFT_DYN_SEQ;
            const int budget = min(P.n_predicts, 1 + (int)((double)d_len * P.alpha));
            endpos = recs[(size_t)d_idx * SAMD_REC + R_END];
            src = text;
            text_n = g.n;
            // [start] + text[e+1 : e+n]  (no padding; samd_sam_only/sam/dyn_sam.py:116-119)
            const int avail = max(0, min(endpos + budget, text_n + 1) - (endpos + 1));
            n_out = 1 + avail;
        } else {
            type = SAMD_DRAFT_STATIC_TREE;
            n_out = 0;
        }
    }
    if (P.out_draft) {
        int32_t *dr = P.out_draft + (size_t)r * P.draft_stride;
        for (int j = lane; j < P.draft_stride; j += 32) {
            int v = 0;
            if (j < n_out) {
                if (j == 0) v = tok;
                else {
                    const int pos = endpos + j;
                    v = (pos <= text_n) ? src[pos] : 0;       // zero padding past the end of the text
                }
            }
            dr[j] = v;
        }
    }
    if (lane == 0) {
        if (P.out_type) P.out_type[r] = type;
        if (P.out_match_dyn) P.out_match_dyn[r] = d_len;
        if (P.out_match_static) P.out_match_static[r] = t_len;
        if (P.out_index_dyn) P.out_index_dyn[r] = d_idx;
        if (P.out_index_static) P.out_index_static[r] = t_idx;
        if (P.out_draft_len) P.out_draft_len[r] = n_out;
        meta[META_PROBES] += q_hops;          // probes spent in lookups (the extend-side count is META_HOPS)
        if constexpr (kProf) {
            const long long t = clock64();
            const size_t n = (size_t)P.dyn.n_requests;
            const long long v[10] = {t - t_begin, c_transfer, c_append, t - t_lookup, acc[0], acc[1], 0, acc[2], acc[3], acc[4]};
            for (int i = 0; i < 10; ++i) P.dbg_cycles[i * n + r] = v[i];
        }
    }
}


// =======================================================================================================
// Kernel variant 1 (default): one THREAD per request builds, one thread per scout (sam_scalar.cuh).  Same CTA
// shape as above - warp 0 the builder, warp 1 the cursor scout, warp 2 the redirect scout (or, with a static
// automaton attached, the static cursor's scout) - but only lane 0 of every warp walks; the builder's other
// lanes join for the coalesced draft copy.  Every record is four 128-bit loads into one thread's registers, a
// probe is five compares: no ballot / shuffle between a record's arrival and the next address.
// =======================================================================================================
__device__ __forceinline__ bool sc_bad(long long idx, long long cap) { return (unsigned long long)idx >= (unsigned long long)cap; }

// Cursor scout, one thread: transfers only, on the automaton as it is, writes nothing.  The record it loads after a
// hit is the record the builder's append reads at the end of its chain (and the next token's cursor record).
template <bool kStatic>
__device__ __forceinline__ void sc_scout_walk(const int32_t *recs, const uint4 *slots, uint32_t bmask, const int32_t *text,
                                              int idx, const int32_t *tk, int k, int peek, int n_predicts, long long text_n,
                                              long long cap, volatile int *mailbox, int prewalk) {
    if (k > SCOUT_MAX_TOKENS) return;
    if (sc_bad(idx, cap)) return;
    const int total = k + (peek >= 0 ? 1 : 0);
    Rec Y = rec_load<kStatic>(recs, idx);
    int next_tok = total > 0 ? (k > 0 ? tk[0] : peek) : 0;
    for (int i = 0; i < total; ++i) {
        const int tok = next_tok;
        if (i + 1 < total) next_tok = i + 1 < k ? tk[i + 1] : peek;
        int up_state = 0, up_target = 0;
        while (true) {
            const Probe pr = rec_probe<kStatic>(Y, slots, bmask, idx, tok, 16);
            if (pr.found) {
                const int up = Y.w[R_LINK];
                idx = sc_bad(pr.target, cap) ? 0 : pr.target;
                Y = rec_load<kStatic>(recs, idx);
                if (!kStatic && i < k) {
                    // the first stop of a clone's redirect walk: requested without waiting for it
                    if (up > 0 && !sc_bad(up, cap)) sc_prefetch_rec(recs, up);
                    up_state = up;
                    up_target = pr.target;
                }
                break;
            }
            if (idx == 0) break;
            idx = Y.w[R_LINK];
            if (sc_bad(idx, cap)) idx = 0;
            Y = rec_load<kStatic>(recs, idx);
            // the stop's overflow slot for this token, should it turn out to be a hub: its address needs only the state's
            // number, so it is requested together with the record instead of after it
            sc_prefetch(slots + (size_t)(samd_hash((uint32_t)idx, (uint32_t)tok) & bmask) * SAMD_BUCKET);
        }
        if (!kStatic && mailbox && i < k) {                  // every token gets an entry (stop 0 = nothing to look up)
            // (atomics: a hand-off between two warps of the CTA that the race checker can follow)
            atomicExch((int *)&mailbox[4 * i + 0], up_state);
            atomicExch((int *)&mailbox[4 * i + 1], tok);
            atomicExch((int *)&mailbox[4 * i + 2], up_target);
            __threadfence_block();
            atomicExch((int *)&mailbox[4 * SCOUT_MAX_TOKENS], i + 1);
        }
    }
    if (peek < 0) return;
    if (!kStatic && idx != 0) {
        // to_anc (dyn_sam.py:99-105) moves the draft's anchor up the suffix chain while the occurrence is too close to the
        // end of the text: walk it too, so that those records and the RIGHT text lines are what gets requested
        const long long n_after = text_n + k;
        for (int hop = 0; hop < 8 && Y.w[R_LINK] > 0 && !sc_bad(Y.w[R_LINK], cap) && n_predicts > n_after - Y.w[R_END]; ++hop) {
            idx = Y.w[R_LINK];
            Y = rec_load<kStatic>(recs, idx);
        }
    }
    const long long e = Y.w[R_END];                          // the draft is read right after this position
    if (e < 0 || e > text_n) return;
    for (int j = 0; j < n_predicts + 8 && e + 1 + j <= text_n; j += 8) sc_prefetch(text + e + 1 + j);
    // Look-ahead for the NEXT step: the draft is what the next step will most likely be handed as accepted tokens
    // (that is what a draft is), so the cursor's path along it is what the next launch will read first.  Walking it
    // now brings those records into L2 (L1 does not survive the launch): next step's cold misses become L2 hits.
    for (int j = 0; j < prewalk && e + 1 + j <= text_n; ++j) {
        const int tok = kStatic ? __ldg(text + e + 1 + j) : text[e + 1 + j];
        while (true) {
            const Probe pr = rec_probe<kStatic>(Y, slots, bmask, idx, tok, 16);
            if (pr.found) {
                idx = sc_bad(pr.target, cap) ? 0 : pr.target;
                Y = rec_load<kStatic>(recs, idx);
                break;
            }
            if (idx == 0) return;                            // the draft left what the automaton knows
            idx = Y.w[R_LINK];
            if (sc_bad(idx, cap)) return;
            Y = rec_load<kStatic>(recs, idx);
        }
        if (idx == 0) return;
    }
}

__device__ __forceinline__ void sc_redirect_scout(const int32_t *recs, const uint4 *slots, uint32_t bmask, volatile int *mailbox,
                                                  int k, long long cap) {
    if (k > SCOUT_MAX_TOKENS) return;
    for (int i = 0; i < k; ++i) {
        while (true) {
            if (atomicAdd((int *)&mailbox[4 * SCOUT_MAX_TOKENS], 0) > i) break;
            if (atomicAdd((int *)&mailbox[4 * SCOUT_MAX_TOKENS + 1], 0)) return;   // the cursor scout is done and never got this far
            __nanosleep(40);
        }
        __threadfence_block();
        int pp = atomicAdd((int *)&mailbox[4 * i + 0], 0);
        const int tok = atomicAdd((int *)&mailbox[4 * i + 1], 0);
        const int target = atomicAdd((int *)&mailbox[4 * i + 2], 0);
        for (int up = 0; up < 6 && pp > 0 && !sc_bad(pp, cap); ++up) {
            const Rec Y = rec_load<false>(recs, pp);
            const Probe pr = rec_probe<false>(Y, slots, bmask, pp, tok, 16);
            if (!pr.found || pr.target != target) break;
            pp = Y.w[R_LINK];
        }
    }
}

// kStatic = false: the launch has no static automaton (the c2 / c1 shape) - its cursor, its scout and their registers are
// compiled out.
template <bool kProf, bool kStatic>
__device__ __forceinline__ void sam_step_scalar_body(const StepParams &P) {
    const bool has_static = kStatic && P.has_static;
    __shared__ int s_mailbox[4 * SCOUT_MAX_TOKENS + 2];
    const int r = blockIdx.x;
    const int lane = threadIdx.x & 31;
    if (r >= P.dyn.n_requests) return;
    if (threadIdx.x < 2) s_mailbox[4 * SCOUT_MAX_TOKENS + threadIdx.x] = 0;
    __syncthreads();
    int32_t *recs = P.dyn.recs + (size_t)r * P.dyn.s_cap * SAMD_REC;
    uint4 *slots = P.dyn.slots + (size_t)r * P.dyn.h_cap;
    int32_t *text = P.dyn.text + (size_t)r * P.dyn.t_cap;
    int32_t *meta = P.dyn.meta + (size_t)r * META_WORDS;
    if (threadIdx.x >= 32) {
        const int k = P.tokens ? (P.counts ? samd_clamp_count(P.counts[r], P.token_stride) : P.token_stride) : 0;
        const int32_t *tk = P.tokens ? P.tokens + (size_t)r * P.token_stride : nullptr;
        if (lane != 0) {
            // Idle lanes of the third warp, one per token of the step: short-context scouts.  A cursor walk that falls
            // back (the token is new in its long context) ends at the states of the last one, two, three tokens - hubs
            // with overflow lists, the most expensive stops of the chain - or at the root.  Lane j walks from the root
            // through tokens j, j+1, j+2: their records and overflow slots are requested up front, all lanes at once.
            if (threadIdx.x >= 64 && lane <= 8 && lane <= k && k <= SCOUT_MAX_TOKENS && P.ngram >= 0) {
                const long long cap = (long long)P.dyn.s_cap;
                const int i = lane - 1;
                const int peek = P.start_tok ? P.start_tok[r] : -1;
                const int total = k + (peek >= 0 ? 1 : 0);
                Rec Y = rec_load<false>(recs, 0);
                Probe pr = rec_probe<false>(Y, slots, P.dyn.bmask, 0, tk[i], 16);
                int idx = (pr.found && !sc_bad(pr.target, cap)) ? pr.target : 0;
                for (int d = 1; d <= P.ngram && idx != 0 && i + d < total; ++d) {
                    const int tokn = i + d < k ? tk[i + d] : peek;
                    sc_prefetch(slots + (size_t)(samd_hash((uint32_t)idx, (uint32_t)tokn) & P.dyn.bmask) * SAMD_BUCKET);
                    Y = rec_load<false>(recs, idx);
                    pr = rec_probe<false>(Y, slots, P.dyn.bmask, idx, tokn, 16);
                    if (!pr.found || sc_bad(pr.target, cap)) break;
                    idx = pr.target;
                }
                if (idx != 0) sc_prefetch_rec(recs, idx);
            }
            return;
        }
        const int peek = P.start_tok ? P.start_tok[r] : -1;
        if (threadIdx.x < 64 && !(has_static && blockDim.x == 64)) {
            sc_scout_walk<false>(recs, slots, P.dyn.bmask, text, meta[META_CUR], tk, k, peek, P.n_predicts, (long long)meta[META_N],
                                 (long long)P.dyn.s_cap, (blockDim.x > 64 && !has_static) ? s_mailbox : nullptr, P.prewalk);
            __threadfence_block();
            atomicExch(&s_mailbox[4 * SCOUT_MAX_TOKENS + 1], 1);         // whatever path the scout left by: no more hand-offs
        } else if (has_static) {
            sc_scout_walk<true>(P.st.recs, P.st.slots, P.st.bmask, P.st.text, P.static_cursor[2 * r], tk, k, peek, P.n_predicts,
                                (long long)P.st.n_tokens, (long long)P.st.n_states, nullptr, P.prewalk);
        } else {
            sc_redirect_scout(recs, slots, P.dyn.bmask, s_mailbox, k, (long long)P.dyn.s_cap);
        }
        return;
    }
    // ---- warp 0: lane 0 builds and looks up, then the warp copies the draft ----
    int o_have = 0, o_n_out = 0, o_endpos = 0, o_text_n = 0, o_src = 0, o_tok = 0;
    if (lane == 0) {
        const long long t_begin = kProf ? clock64() : 0;
        unsigned long long g_begin = 0;
        if constexpr (kProf) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_begin));
        ScBuilderT<kProf> b;
        if constexpr (kProf)
            for (int i = 0; i < SC_PF_N; ++i) b.pf[i] = 0;
        // the arena's base pointers stay in registers (otherwise every address is rebuilt from the constant bank)
        asm volatile("" : "+l"(recs), "+l"(slots));
        b.d.recs = recs;
        b.d.slots = slots;
        b.d.text = text;
        {
            unsigned bm = P.dyn.bmask;                        // (likewise: not re-read from the constant bank at every use)
            int mt = P.dyn.max_tokens;
            asm volatile("" : "+r"(bm), "+r"(mt));
            b.d.bmask = bm;
            b.d.max_tokens = mt;
        }
        b.x_state = -1;
        b.tr.trace = (kProf && P.trace) ? P.trace + (size_t)r * P.trace_cap + 1 : nullptr;
        b.tr.cap = P.trace_cap - 1;
        b.tr.n = 0;
        // every input of the step is requested at once: the meta block, the step's first token, its count, the lookup
        // token and the static cursor are independent loads - one round trip instead of a chain of them
        const int32_t *tk = P.tokens ? P.tokens + (size_t)r * P.token_stride : nullptr;
        int lookup_probes;
        int next_tok = 0, k = 0, start_tok = 0, s_idx = 0, s_len = 0, s_hops = 0;
        {
            const int4 m0 = *reinterpret_cast<const int4 *>(meta), m1 = *reinterpret_cast<const int4 *>(meta + 4);
            const int4 m2 = *reinterpret_cast<const int4 *>(meta + 8), m3 = *reinterpret_cast<const int4 *>(meta + 12);
            if (tk) {
                next_tok = tk[0];
                k = P.counts ? samd_clamp_count(P.counts[r], P.token_stride) : P.token_stride;
            }
            if (P.start_tok) start_tok = P.start_tok[r];
            if (has_static) {
                s_idx = P.static_cursor[2 * r];
                s_len = P.static_cursor[2 * r + 1];
            }
            b.g.n_states = m0.x; b.g.last = m0.y; b.g.n = m0.z; b.g.cur = m0.w;
            b.g.cur_len = m1.x; b.g.n_edges = m1.y; b.g.n_clones = m1.w;
            b.g.hops = m2.x; lookup_probes = m2.y; b.g.last_link = m2.z; b.g.ll_twin = m2.w;
            b.g.ll_len = m3.x; b.g.ll_link = m3.y; b.g.max_chain = m3.z;
        }
        const long long t_tokens = kProf ? clock64() : 0;
        // ---- phase 1: DraftModel.update (draft.py:65-79) ----
        if (P.tokens) {
            int flags = 0;
            for (int i = 0; i < k; ++i) {
                const int tok = next_tok;
                if (i + 1 < k) next_tok = tk[i + 1];         // one ahead: the next token is in a register when its turn comes
                if (tok < 0) {                               // -1 marks a free edge slot in the layout: never a token
                    flags |= 2;
                    break;
                }
                if (has_static) sc_prefetch_rec(P.st.recs, s_idx);
                if (b.g.n >= b.d.max_tokens) {
                    // arena full: the token cannot be appended (the flag tells the caller to grow); the cursors still
                    // follow the text so that the lookups keep returning what the automaton knows
                    flags |= 1;
                    b.transfer_one(tok);
                } else {
                    b.extend_one(tok);                       // add_tokens: match first, then append (dyn_sam.py:84-88)
                }
                if (has_static) sc_transfer<true>(P.st.recs, P.st.slots, P.st.bmask, s_idx, s_len, tok, s_hops);
            }
            *reinterpret_cast<int4 *>(meta) = make_int4(b.g.n_states, b.g.last, b.g.n, b.g.cur);
            meta[META_CURLEN] = b.g.cur_len;
            meta[META_NEDGES] = b.g.n_edges;
            meta[META_NCLONES] = b.g.n_clones;
            meta[META_HOPS] = b.g.hops;
            meta[META_LASTLINK] = b.g.last_link;
            meta[META_LLTWIN] = b.g.ll_twin;
            meta[META_LLLEN] = b.g.ll_len;
            meta[META_LLLINK] = b.g.ll_link;
            meta[META_MAXCHAIN] = b.g.max_chain;
            if (flags) meta[META_OVERFLOW] |= flags;
            if (has_static) {
                P.static_cursor[2 * r] = s_idx;
                P.static_cursor[2 * r + 1] = s_len;
            }
        }
        const long long t_lookup = kProf ? clock64() : 0;
        // ---- phase 2: DraftModel.lookup (draft.py:52-63 / samd_sam_only/draft.py:49-59) ----
        if (P.start_tok) {
            const int tok = start_tok;
            int d_idx = 0, d_len = 0, q_hops = 0;
            b.lookup(tok, d_idx, d_len, q_hops);
            int t_idx = 0, t_len = 0;
            if (has_static) {
                t_idx = s_idx;
                t_len = s_len;
                sc_transfer<true>(P.st.recs, P.st.slots, P.st.bmask, t_idx, t_len, tok, s_hops);
            }
            const int t_biased = t_len - P.len_bias;
            int type, n_out, endpos = 0, text_n = 0, src = 0;
            if (P.flavour == SAMD_FLAVOUR_SAMD) {
                n_out = P.n_predicts;
                if (max(d_len, t_biased) >= P.len_threshold) {
                    if (d_len >= t_biased) {
                        type = SAMD_DRAFT_DYN_SEQ;
                        endpos = b.anchor_samd(d_idx, P.n_predicts);         // to_anc (dyn_sam.py:99-105)
                        text_n = b.g.n;
                    } else {
                        type = SAMD_DRAFT_STATIC_SEQ;
                        endpos = __ldg(P.st.recs + (size_t)t_idx * SAMD_REC + R_END);
                        src = 1;
                        text_n = (int)P.st.n_tokens;
                    }
                } else {
                    type = SAMD_DRAFT_TREE_MODEL;
                    n_out = 0;
                }
            } else {
                if (d_len >= t_biased) {
                    type = SAMD_DRAFT_DYN_SEQ;
                    const int budget = min(P.n_predicts, 1 + (int)((double)d_len * P.alpha));
                    endpos = recs[(size_t)d_idx * SAMD_REC + R_END];
                    text_n = b.g.n;
                    // [start] + text[e+1 : e+n]  (no padding; samd_sam_only/sam/dyn_sam.py:116-119)
                    n_out = 1 + max(0, min(endpos + budget, text_n + 1) - (endpos + 1));
                } else {
                    type = SAMD_DRAFT_STATIC_TREE;
                    n_out = 0;
                }
            }
            if (P.out_type) P.out_type[r] = type;
            if (P.out_match_dyn) P.out_match_dyn[r] = d_len;
            if (P.out_match_static) P.out_match_static[r] = t_len;
            if (P.out_index_dyn) P.out_index_dyn[r] = d_idx;
            if (P.out_index_static) P.out_index_static[r] = t_idx;
            if (P.out_draft_len) P.out_draft_len[r] = n_out;
            meta[META_PROBES] = lookup_probes + q_hops;
            o_have = 1; o_n_out = n_out; o_endpos = endpos; o_text_n = text_n; o_src = src; o_tok = tok;
        }
        if constexpr (kProf)
            if (b.tr.trace) b.tr.trace[-1] = b.tr.n;
        if constexpr (kProf) {
            if (P.start_tok) {
                const long long t = clock64();
                const size_t n = (size_t)P.dyn.n_requests;
                // whole request, cycles waiting for record loads, update phase, lookup phase, record loads that took
                // < 120 / < 500 / < 1100 / more cycles (L1 / L2 / DRAM / slower), overflow-probe cycles and count
                const long long v[10] = {t - t_begin, b.pf[SC_PF_LOAD_CYC], t_lookup - t_begin, t - t_lookup, b.pf[SC_PF_L1], b.pf[SC_PF_L2],
                                         b.pf[SC_PF_DRAM], b.pf[SC_PF_SLOW], b.pf[SC_PF_OVF_CYC], b.pf[SC_PF_OVF_N]};
                for (int i = 0; i < 10; ++i) P.dbg_cycles[i * n + r] = v[i];
                unsigned long long g1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
                P.dbg_cycles[10 * n + r] = (long long)g_begin;       // ns, comparable across SMs: the step's span
                P.dbg_cycles[11 * n + r] = (long long)g1;
                P.dbg_cycles[12 * n + r] = b.pf[SC_PF_WALK_CYC];     // cursor walks (incl. fused inserts), clone redirect walks,
                P.dbg_cycles[13 * n + r] = b.pf[SC_PF_REDIR_CYC];    // cycles before the first token starts
                P.dbg_cycles[14 * n + r] = t_tokens - t_begin;
                P.dbg_cycles[15 * n + r] = b.pf[SC_PF_REDIR_N];      // records read by the redirect walks
            }
        }
    }
    __syncwarp();
    o_have = __shfl_sync(SAMD_FULL, o_have, 0);
    if (!o_have || !P.out_draft) return;
    o_n_out = __shfl_sync(SAMD_FULL, o_n_out, 0);
    o_endpos = __shfl_sync(SAMD_FULL, o_endpos, 0);
    o_text_n = __shfl_sync(SAMD_FULL, o_text_n, 0);
    o_src = __shfl_sync(SAMD_FULL, o_src, 0);
    o_tok = __shfl_sync(SAMD_FULL, o_tok, 0);
    const int32_t *src = o_src ? P.st.text : text;
    int32_t *dr = P.out_draft + (size_t)r * P.draft_stride;
    for (int j = lane; j < P.draft_stride; j += 32) {
        int v = 0;
        if (j < o_n_out) {
            if (j == 0) v = o_tok;
            else {
                const int pos = o_endpos + j;
                v = (pos <= o_text_n) ? src[pos] : 0;         // zero padding past the end of the text
            }
        }
        dr[j] = v;
    }
}

// Three builds of the same body: the wide one with a static automaton (three warps, capped at 96 registers: six CTAs per
// SM), the dynamic-only one below (80 registers: eight CTAs per SM), and a lean one (64 registers, two warps: 16 CTAs per
// SM) for batches so large that residency matters more than the third warp - 4096 static-SAM cursors (config c3) would
// otherwise run in four waves.
#ifndef SAMD_STEP_DYN_REGS
#define SAMD_STEP_DYN_REGS 80
#endif
template <bool kProf>
__global__ void __maxnreg__(96) sam_step_scalar_kernel(StepParams P) {
    sam_step_scalar_body<kProf, true>(P);
}
// The dynamic-automaton-only build at 80 registers: a warp of 96-register threads takes 3072 registers of a 16384-register
// scheduler partition, so only five fit (20 warps = SIX three-warp CTAs per SM, 888 requests per wave - ncu's
// launch__occupancy_limit_registers - and the 136 late CTAs of a 1024-request step start when the first short requests are
// done: 16.7 us); at 80 registers six warps fit, eight CTAs per SM, and the whole batch is resident at once.
__global__ void __maxnreg__(SAMD_STEP_DYN_REGS) sam_step_scalar_dyn_kernel(StepParams P) {
    sam_step_scalar_body<false, false>(P);
}
__global__ void __maxnreg__(64) sam_step_scalar_lean_kernel(StepParams P) {
    sam_step_scalar_body<false, true>(P);
}

static long long *g_dbg_cycles = nullptr;
static int g_scouts = 2;
static int g_variant = 1;
static int g_prewalk = 0;
static int g_ngram = 6;
static int g_lean = -1;
static int32_t *g_trace = nullptr;
static int g_trace_cap = 0;
extern "C" void samd_step_set_scouts(int on) { g_scouts = on; }
extern "C" void samd_step_set_variant(int v) { g_variant = v; }
extern "C" void samd_step_set_prewalk(int n) { g_prewalk = n < 0 ? 0 : n; }
extern "C" void samd_step_set_ngram(int depth) { g_ngram = depth; }
extern "C" void samd_step_set_lean(int mode) { g_lean = mode; }
extern "C" void samd_step_set_trace(int32_t *trace_dev, int cap) {
    g_trace = trace_dev;
    g_trace_cap = trace_dev ? cap : 0;
}
extern "C" void samd_step_set_debug_cycles(int64_t *cycles_dev) { g_dbg_cycles = (long long *)cycles_dev; }

// The host-buffer path's staging copy as a KERNEL: 16-byte coalesced loads turn into a few hundred full-size PCIe read
// requests when `src` is mapped pinned host memory, where the step kernel's own per-request reads (a 4-byte count, a
// 32-byte token row and a start token per CTA, repeated by its scouts) are thousands of small non-posted reads.  A
// copy-engine memcpy node in the same graph costs ~10 us more per step than this launch (DESIGN.md section 5).
__global__ void __launch_bounds__(256) stage_copy_kernel(uint4 *__restrict__ dst, const uint4 *__restrict__ src, long long n16,
                                                         int32_t *__restrict__ dst_w, const int32_t *__restrict__ src_w, int n_tail) {
    const long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long i = i0; i < n16; i += (long long)gridDim.x * blockDim.x) dst[i] = src[i];
    if (i0 < n_tail) dst_w[i0] = src_w[i0];
}

extern "C" int samd_stage_copy(void *dst, const void *src, int64_t n_bytes, void *stream) {
    SAMD_REQUIRE(dst && src && n_bytes >= 0, "samd_stage_copy: bad arguments");
    SAMD_REQUIRE(((uintptr_t)dst & 15) == 0 && ((uintptr_t)src & 15) == 0 && (n_bytes & 3) == 0,
                 "samd_stage_copy: pointers must be 16-byte aligned and the size a multiple of 4");
    if (n_bytes == 0) return 0;
    const long long n16 = n_bytes >> 4;
    const int n_tail = (int)((n_bytes & 15) >> 2);
    long long blocks = (n16 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 592) blocks = 592;
    stage_copy_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>((uint4 *)dst, (const uint4 *)src, n16, (int32_t *)dst + 4 * n16,
                                                                    (const int32_t *)src + 4 * n16, n_tail);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int samd_step(const samd_step_args *a, void *stream) {
    SAMD_REQUIRE(a && a->dyn, "samd_step: dyn handle required");
    SAMD_REQUIRE((a->stat == nullptr) == (a->static_cursor_dev == nullptr),
                 "samd_step: static handle and static cursor must be given together");
    SAMD_REQUIRE(!a->stat || a->stat->dev.recs, "samd_step: static automaton is not on the device");
    StepParams P;
    P.dyn = a->dyn->a;
    P.has_static = a->stat != nullptr;
    if (a->stat) P.st = a->stat->dev;
    else P.st = StaticDev{};
    P.static_cursor = a->static_cursor_dev;
    P.tokens = a->tokens_dev;
    P.token_stride = a->token_stride;
    P.counts = a->counts_dev;
    P.start_tok = a->start_tok_dev;
    P.flavour = a->flavour;
    P.n_predicts = a->n_predicts;
    P.len_bias = a->len_bias;
    P.len_threshold = a->len_threshold;
    P.alpha = a->alpha;
    P.out_type = a->out_type_dev;
    P.out_match_dyn = a->out_match_dyn_dev;
    P.out_match_static = a->out_match_static_dev;
    P.out_index_dyn = a->out_index_dyn_dev;
    P.out_index_static = a->out_index_static_dev;
    P.out_draft = a->out_draft_dev;
    P.out_draft_len = a->out_draft_len_dev;
    P.draft_stride = a->draft_stride;
    P.dbg_cycles = g_dbg_cycles;
    P.prewalk = g_prewalk;
    P.ngram = g_ngram;
    P.trace = g_trace;
    P.trace_cap = g_trace_cap;
    SAMD_REQUIRE(a->flavour == SAMD_FLAVOUR_SAMD || a->flavour == SAMD_FLAVOUR_SAM_ONLY, "samd_step: bad flavour");
    SAMD_REQUIRE(!a->tokens_dev || a->token_stride > 0, "samd_step: token_stride must be positive");
    SAMD_REQUIRE(!a->out_draft_dev || a->draft_stride >= a->n_predicts, "samd_step: draft_stride < n_predicts");
    // warp 0 builds, warp 1 scouts the dynamic automaton, warp 2 the static one (if any), warp 3 the clones' redirect walks
    // (with a static automaton the redirect scout is left out: measured on c3, 4096 mostly static-drafting requests, it
    // costs more than it brings - 49.2 vs 43.2 us per step)
    if (g_variant == 1) {
        // builder + cursor scout + (static cursor scout | redirect scout); one walking thread per warp
        int threads = g_scouts ? ((P.has_static || (a->tokens_dev && g_scouts > 1)) ? 96 : 64) : 32;
        static int n_sm = 0;
        if (!n_sm) {
            int dev = 0;
            SAMD_CUDA(cudaGetDevice(&dev));
            SAMD_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        }
        // more requests than one wave of the wide build (eight CTAs per SM without a static automaton, six with one)
        const bool lean = g_lean >= 0 ? g_lean != 0 : P.dyn.n_requests > (P.has_static ? 6 : 8) * n_sm;
        if (lean && threads > 64) threads = 64;
        if (P.dbg_cycles) sam_step_scalar_kernel<true><<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
        else if (lean) sam_step_scalar_lean_kernel<<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
        else if (!P.has_static) sam_step_scalar_dyn_kernel<<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
        else sam_step_scalar_kernel<false><<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
        samd_count_launch();
        SAMD_CUDA(cudaGetLastError());
        return 0;
    }
    const int threads = g_scouts ? (P.has_static ? 96 : (a->tokens_dev && g_scouts > 1 ? 128 : 64)) : 32;
    if (P.dbg_cycles) sam_step_kernel<true><<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
    else sam_step_kernel<false><<<P.dyn.n_requests, threads, 0, (cudaStream_t)stream>>>(P);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// document-sharded static SAM: per-shard packed keys, draft from the winning global position
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) static_keys_kernel(StaticDev st, const int32_t *cursor, const int32_t *start_tok,
                                                         int n, long long shard_offset, long long *keys) {
    const int r = blockIdx.x;
    const int lane = threadIdx.x;
    if (r >= n) return;
    int idx = cursor[2 * r], len = cursor[2 * r + 1];
    int hops = 0;
    warp_transfer<true>(st.recs, st.slots, st.bmask, idx, len, start_tok[r], lane, hops);
    if (lane == 0) {
        long long key = 0;
        if (len > 0) {
            const long long e = shard_offset + (long long)__ldg(st.recs + (size_t)idx * SAMD_REC + R_END);
            key = ((long long)len << 32) | (long long)(0xFFFFFFFFu - (uint32_t)e);
        }
        keys[r] = key;
    }
}

extern "C" int samd_static_lookup_keys(samd_static_t h, const int32_t *static_cursor_dev, const int32_t *start_tok_dev,
                                       int n_requests, int64_t shard_offset, int64_t *out_keys_dev, void *stream) {
    SAMD_REQUIRE(h && h->dev.recs && static_cursor_dev && start_tok_dev && out_keys_dev && n_requests > 0,
                 "samd_static_lookup_keys: bad arguments");
    static_keys_kernel<<<n_requests, 32, 0, (cudaStream_t)stream>>>(h->dev, static_cursor_dev, start_tok_dev, n_requests,
                                                                     (long long)shard_offset, (long long *)out_keys_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

__global__ void draft_from_keys_kernel(const long long *keys, const int32_t *corpus, long long n_tokens,
                                       const int32_t *start_tok, int n, int n_predicts, int32_t *out_match, int32_t *out_draft,
                                       int stride) {
    const int r = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (r >= n) return;
    const long long key = keys[r];
    const int len = (int)(key >> 32);
    // no match anywhere: endpos 0 (root), like StaticSAM.gen_draft on index 0 (static_sam.py:119-125)
    const long long e = len > 0 ? (long long)(0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFll)) : 0;
    if (lane == 0 && out_match) out_match[r] = len;
    for (int j = lane; j < stride; j += 32) {
        int v = 0;
        if (j < n_predicts) {
            if (j == 0) v = start_tok[r];
            else {
                const long long pos = e + j;
                v = pos <= n_tokens ? corpus[pos] : 0;
            }
        }
        out_draft[(size_t)r * stride + j] = v;
    }
}

extern "C" int samd_draft_from_keys(const int64_t *keys_dev, const int32_t *corpus_dev, int64_t n_corpus_tokens,
                                    const int32_t *start_tok_dev, int n_requests, int32_t n_predicts, int32_t *out_match_dev,
                                    int32_t *out_draft_dev, int32_t draft_stride, void *stream) {
    SAMD_REQUIRE(keys_dev && corpus_dev && start_tok_dev && out_draft_dev && n_requests > 0 && draft_stride >= n_predicts,
                 "samd_draft_from_keys: bad arguments");
    const int wpb = 8;
    draft_from_keys_kernel<<<(n_requests + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(
        (const long long *)keys_dev, corpus_dev, (long long)n_corpus_tokens, start_tok_dev, n_requests, n_predicts,
        out_match_dev, out_draft_dev, draft_stride);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// stand-alone gen_draft entry points (the drop-in DynSAM.gen_draft / StaticSAM.gen_draft may be
// called with any state index, not only the one the last lookup returned)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) dyn_gen_draft_kernel(DynArena a, const int32_t *index, const int32_t *match,
                                                           const int32_t *start_tok, int flavour, int n_predicts, double alpha,
                                                           int32_t *out_draft, int stride, int32_t *out_len) {
    const int r = blockIdx.x, lane = threadIdx.x;
    if (r >= a.n_requests) return;
    const int32_t *recs = a.recs + (size_t)r * a.s_cap * SAMD_REC;
    const int32_t *text = a.text + (size_t)r * a.t_cap;
    const int n = a.meta[(size_t)r * META_WORDS + META_N];
    int idx = index[r];
    int4 rec = *reinterpret_cast<const int4 *>(recs + (size_t)idx * SAMD_REC);
    int n_out;
    if (flavour == SAMD_FLAVOUR_SAMD) {
        if (idx != 0) {                                      // to_anc (dyn_sam.py:99-105)
            while (rec.x != 0 && n_predicts > n - rec.z) {
                idx = rec.x;
                rec = *reinterpret_cast<const int4 *>(recs + (size_t)idx * SAMD_REC);
            }
        }
        n_out = n_predicts;
    } else {
        const int budget = min(n_predicts, 1 + (int)((double)match[r] * alpha));
        n_out = 1 + max(0, min(rec.z + budget, n + 1) - (rec.z + 1));
    }
    for (int j = lane; j < stride; j += 32) {
        int v = 0;
        if (j < n_out) v = j == 0 ? start_tok[r] : (rec.z + j <= n ? text[rec.z + j] : 0);
        out_draft[(size_t)r * stride + j] = v;
    }
    if (lane == 0 && out_len) out_len[r] = n_out;
}

extern "C" int samd_dyn_gen_draft(samd_dyn_t h, const int32_t *index_dev, const int32_t *match_dev, const int32_t *start_tok_dev,
                                  int32_t flavour, int32_t n_predicts, double alpha, int32_t *out_draft_dev, int32_t draft_stride,
                                  int32_t *out_len_dev, void *stream) {
    SAMD_REQUIRE(h && index_dev && start_tok_dev && out_draft_dev && draft_stride >= n_predicts, "samd_dyn_gen_draft: bad arguments");
    SAMD_REQUIRE(flavour == SAMD_FLAVOUR_SAMD || match_dev, "samd_dyn_gen_draft: sam_only flavour needs match lengths");
    dyn_gen_draft_kernel<<<h->a.n_requests, 32, 0, (cudaStream_t)stream>>>(h->a, index_dev, match_dev, start_tok_dev, flavour,
                                                                             n_predicts, alpha, out_draft_dev, draft_stride, out_len_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

__global__ void static_gen_draft_kernel(StaticDev st, const int32_t *index, const int32_t *start_tok, int n, int n_predicts,
                                        int32_t *out_draft, int stride) {
    const int r = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x & 31;
    if (r >= n) return;
    const int e = __ldg(st.recs + (size_t)index[r] * SAMD_REC + R_END);   // static_sam.py:119-125 (no to_anc)
    for (int j = lane; j < stride; j += 32) {
        int v = 0;
        if (j < n_predicts) v = j == 0 ? start_tok[r] : ((long long)e + j <= st.n_tokens ? st.text[e + j] : 0);
        out_draft[(size_t)r * stride + j] = v;
    }
}

extern "C" int samd_static_gen_draft(samd_static_t h, const int32_t *index_dev, const int32_t *start_tok_dev, int n_requests,
                                     int32_t n_predicts, int32_t *out_draft_dev, int32_t draft_stride, void *stream) {
    SAMD_REQUIRE(h && h->dev.recs && index_dev && start_tok_dev && out_draft_dev && n_requests > 0 && draft_stride >= n_predicts,
                 "samd_static_gen_draft: bad arguments");
    static_gen_draft_kernel<<<(n_requests + 7) / 8, 256, 0, (cudaStream_t)stream>>>(h->dev, index_dev, start_tok_dev, n_requests,
                                                                                    n_predicts, out_draft_dev, draft_stride);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// out-edges of state v in insertion order: inline edges, then the overflow list (oldest first)
template <class F>
static inline void host_for_each_edge(const int32_t *recs, const uint4 *slots, int64_t v, F f) {
    const int32_t *rec = recs + (size_t)v * SAMD_REC;
    for (int i = 0; i < SAMD_INLINE && (uint32_t)rec[R_TOK + i] != SAMD_EMPTY; ++i) f(rec[R_TOK + i], rec[R_TGT + i]);
    for (uint32_t e = (uint32_t)rec[R_OHEAD]; e != SAMD_NIL; e = slots[e].w) f((int32_t)slots[e].y, (int32_t)slots[e].z);
}

// edges of one request as (state, token, target) triples, per state in insertion order (oldest first)
extern "C" int samd_dyn_export_edges(samd_dyn_t h, int request, int32_t *edges_host, int64_t capacity) {
    SAMD_REQUIRE(h && request >= 0 && request < h->a.n_requests && edges_host, "samd_dyn_export_edges: bad arguments");
    SAMD_CUDA(cudaDeviceSynchronize());
    int32_t meta[META_WORDS];
    SAMD_CUDA(cudaMemcpy(meta, h->a.meta + (size_t)request * META_WORDS, sizeof(meta), cudaMemcpyDeviceToHost));
    SAMD_REQUIRE(capacity >= meta[META_NEDGES], "samd_dyn_export_edges: capacity too small");
    const int ns = meta[META_NSTATES];
    int32_t *st = (int32_t *)malloc((size_t)ns * SAMD_REC * sizeof(int32_t));
    uint4 *sl = (uint4 *)malloc((size_t)h->a.h_cap * sizeof(uint4));
    SAMD_CUDA(cudaMemcpy(st, h->a.recs + (size_t)request * h->a.s_cap * SAMD_REC, (size_t)ns * SAMD_REC * sizeof(int32_t),
                         cudaMemcpyDeviceToHost));
    SAMD_CUDA(cudaMemcpy(sl, h->a.slots + (size_t)request * h->a.h_cap, (size_t)h->a.h_cap * sizeof(uint4), cudaMemcpyDeviceToHost));
    int64_t k = 0;
    for (int v = 0; v < ns; ++v)
        host_for_each_edge(st, sl, v, [&](int32_t tok, int32_t tgt) {
            if (k < capacity) {
                edges_host[3 * k] = v;
                edges_host[3 * k + 1] = tok;
                edges_host[3 * k + 2] = tgt;
            }
            k++;
        });
    free(st);
    free(sl);
    SAMD_REQUIRE(k == meta[META_NEDGES], "samd_dyn_export_edges: edge count mismatch (corrupt arena)");
    return 0;
}

// ---------------------------------------------------------------------------------------
// cursor-only walks: DynSAM.transfer_tokens (dyn_sam.py:90-92), StaticSAM.transfer_tokens
// (static_sam.py:102-104) and the stand-alone StaticSAM.lookup / DynSAM.lookup (:94-97, :106-109)
// ---------------------------------------------------------------------------------------
template <bool kReadOnly>
__device__ __forceinline__ void cursor_walk(const int32_t *recs, const uint4 *slots, uint32_t bmask, int &idx, int &len,
                                            const int32_t *tk, int k, int lane) {
    int hops = 0;
    for (int i = 0; i < k; i += 32) {
        const int mine = (i + lane < k) ? tk[i + lane] : 0;
        const int lim = min(32, k - i);
        for (int j = 0; j < lim; ++j)
            warp_transfer<kReadOnly>(recs, slots, bmask, idx, len, __shfl_sync(SAMD_FULL, mine, j), lane, hops);
    }
}

__global__ void __launch_bounds__(32) static_walk_kernel(StaticDev st, int32_t *cursor, const int32_t *tokens, int stride,
                                                         const int32_t *counts, const int32_t *peek_tok, int n,
                                                         int32_t *out_index, int32_t *out_len) {
    const int r = blockIdx.x, lane = threadIdx.x;
    if (r >= n) return;
    int idx = cursor[2 * r], len = cursor[2 * r + 1];
    if (tokens) {
        cursor_walk<true>(st.recs, st.slots, st.bmask, idx, len, tokens + (size_t)r * stride, counts ? samd_clamp_count(counts[r], stride) : stride, lane);
        if (lane == 0) {
            cursor[2 * r] = idx;
            cursor[2 * r + 1] = len;
        }
    }
    if (peek_tok) {
        int hops = 0;
        warp_transfer<true>(st.recs, st.slots, st.bmask, idx, len, peek_tok[r], lane, hops);
        if (lane == 0) {
            out_index[r] = idx;
            out_len[r] = len;
        }
    }
}

extern "C" int samd_static_walk(samd_static_t h, int32_t *static_cursor_dev, const int32_t *tokens_dev, int32_t token_stride,
                                const int32_t *counts_dev, const int32_t *peek_tok_dev, int n_requests, int32_t *out_index_dev,
                                int32_t *out_len_dev, void *stream) {
    SAMD_REQUIRE(h && h->dev.recs && static_cursor_dev && n_requests > 0, "samd_static_walk: bad arguments");
    SAMD_REQUIRE(!peek_tok_dev || (out_index_dev && out_len_dev), "samd_static_walk: peek needs output arrays");
    static_walk_kernel<<<n_requests, 32, 0, (cudaStream_t)stream>>>(h->dev, static_cursor_dev, tokens_dev, token_stride, counts_dev,
                                                                     peek_tok_dev, n_requests, out_index_dev, out_len_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

__global__ void __launch_bounds__(32) dyn_walk_kernel(DynArena a, const int32_t *tokens, int stride, const int32_t *counts) {
    const int r = blockIdx.x, lane = threadIdx.x;
    if (r >= a.n_requests) return;
    int32_t *meta = a.meta + (size_t)r * META_WORDS;
    int idx = meta[META_CUR], len = meta[META_CURLEN];
    cursor_walk<false>(a.recs + (size_t)r * a.s_cap * SAMD_REC, a.slots + (size_t)r * a.h_cap, a.bmask, idx, len,
                       tokens + (size_t)r * stride, counts ? samd_clamp_count(counts[r], stride) : stride, lane);
    if (lane == 0) {
        meta[META_CUR] = idx;
        meta[META_CURLEN] = len;
    }
}

extern "C" int samd_dyn_transfer(samd_dyn_t h, const int32_t *tokens_dev, int32_t token_stride, const int32_t *counts_dev,
                                 void *stream) {
    SAMD_REQUIRE(h && tokens_dev && token_stride > 0, "samd_dyn_transfer: bad arguments");
    dyn_walk_kernel<<<h->a.n_requests, 32, 0, (cudaStream_t)stream>>>(h->a, tokens_dev, token_stride, counts_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------
// Capacity growth: a new batch with a larger max_tokens holding the same automata (same state
// numbering, cursor and history).  Records / text / meta are copied; the overflow table is
// re-hashed on the host for the new capacity, keeping every state's edge order.  Rare.
// ---------------------------------------------------------------------------------------
extern "C" int samd_dyn_grow(samd_dyn_t old, int new_max_tokens, samd_dyn_t *out) {
    SAMD_REQUIRE(old && out && new_max_tokens > old->a.max_tokens, "samd_dyn_grow: new capacity must be larger");
    samd_dyn_s *nw = nullptr;
    int rc = samd_dyn_create(old->a.n_requests, new_max_tokens, &nw);
    if (rc) return rc;
    SAMD_CUDA(cudaDeviceSynchronize());
    const DynArena &o = old->a;
    const DynArena &n = nw->a;
    int32_t *st = (int32_t *)malloc((size_t)o.s_cap * SAMD_REC * sizeof(int32_t));
    uint4 *sl = (uint4 *)malloc((size_t)o.h_cap * sizeof(uint4));
    uint4 *nsl = (uint4 *)malloc((size_t)n.h_cap * sizeof(uint4));
    int32_t meta[META_WORDS];
    SAMD_REQUIRE(st && sl && nsl, "samd_dyn_grow: host allocation failed");
    for (int r = 0; r < o.n_requests; ++r) {
        SAMD_CUDA(cudaMemcpy(meta, o.meta + (size_t)r * META_WORDS, sizeof(meta), cudaMemcpyDeviceToHost));
        const int ns = meta[META_NSTATES];
        SAMD_CUDA(cudaMemcpy(st, o.recs + (size_t)r * o.s_cap * SAMD_REC, (size_t)ns * SAMD_REC * sizeof(int32_t), cudaMemcpyDeviceToHost));
        SAMD_CUDA(cudaMemcpy(sl, o.slots + (size_t)r * o.h_cap, (size_t)o.h_cap * sizeof(uint4), cudaMemcpyDeviceToHost));
        memset(nsl, 0xFF, (size_t)n.h_cap * sizeof(uint4));
        for (int v = 0; v < ns; ++v) {
            int32_t *rec = st + (size_t)v * SAMD_REC;
            uint32_t head = SAMD_NIL, tail = SAMD_NIL;
            for (uint32_t e = (uint32_t)rec[R_OHEAD]; e != SAMD_NIL; e = sl[e].w) {     // oldest first
                const uint4 ed = sl[e];
                uint32_t b = samd_hash((uint32_t)v, ed.y) & n.bmask;
                uint32_t slot = 0;
                for (bool placed = false; !placed; b = (b + 1) & n.bmask)
                    for (int l = 0; l < SAMD_BUCKET && !placed; ++l)
                        if (nsl[(size_t)b * SAMD_BUCKET + l].x == SAMD_EMPTY) {
                            slot = b * SAMD_BUCKET + l;
                            placed = true;
                        }
                nsl[slot] = make_uint4((uint32_t)v, ed.y, ed.z, SAMD_NIL);
                if (tail != SAMD_NIL) nsl[tail].w = slot;
                else head = slot;
                tail = slot;
            }
            rec[R_OHEAD] = (int32_t)head;
            rec[R_OTAIL] = (int32_t)tail;
        }
        SAMD_CUDA(cudaMemcpy(n.recs + (size_t)r * n.s_cap * SAMD_REC, st, (size_t)ns * SAMD_REC * sizeof(int32_t), cudaMemcpyHostToDevice));
        SAMD_CUDA(cudaMemcpy(n.slots + (size_t)r * n.h_cap, nsl, (size_t)n.h_cap * sizeof(uint4), cudaMemcpyHostToDevice));
        SAMD_CUDA(cudaMemcpy(n.text + (size_t)r * n.t_cap, o.text + (size_t)r * o.t_cap, (size_t)(meta[META_N] + 1) * sizeof(int32_t),
                             cudaMemcpyDeviceToDevice));
        meta[META_OVERFLOW] = 0;
        SAMD_CUDA(cudaMemcpy(n.meta + (size_t)r * META_WORDS, meta, sizeof(meta), cudaMemcpyHostToDevice));
    }
    free(st);
    free(sl);
    free(nsl);
    *out = nw;
    return 0;
}

// ---------------------------------------------------------------------------------------
// Floor of the step's dependent-load chain (profiling aid, tools/step_floor.py): replay a request's recorded
// sequence of record reads as bare loads, each address made to depend on the previous load's value.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) replay_trace_kernel(DynArena a, const int32_t *trace, int cap, long long *cycles) {
    const int r = blockIdx.x;
    if (r >= a.n_requests || (threadIdx.x & 31) != 0) return;
    const int32_t *recs = a.recs + (size_t)r * a.s_cap * SAMD_REC;
    const int32_t *tr = trace + (size_t)r * cap;
    const int n = min(tr[0], cap - 1);
    if (threadIdx.x >= 32) {                               // the ideal scout: the same records, independent loads
        for (int i = 0; i < n; ++i) {
            const int s = tr[1 + i];
            if (!sc_bad(s, a.s_cap)) sc_prefetch_rec(recs, s);
        }
        return;
    }
    unsigned long long g0, g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g0));
    const long long t0 = clock64();
    int acc = 0;
    for (int i = 0; i < n; ++i) {
        const int s = tr[1 + i] + (acc & 0x40000000);      // always + 0 (a record's length is < 2^28 and its last word 0), but the compiler cannot know
        const Rec Y = rec_load<false>(recs, sc_bad(s, a.s_cap) ? 0 : s);
        acc = (Y.w[R_LEN] & 0x0FFFFFFF) | Y.w[R_AUX];
    }
    const long long dt = clock64() - t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    const size_t nr = (size_t)a.n_requests;
    cycles[r] = dt + (acc & 0x40000000);
    cycles[nr + r] = (long long)g0;
    cycles[2 * nr + r] = (long long)g1;
}

extern "C" int samd_debug_replay_trace(samd_dyn_t h, const int32_t *trace_dev, int cap, int with_scout, int64_t *cycles_dev,
                                       void *stream) {
    SAMD_REQUIRE(h && trace_dev && cap > 1 && cycles_dev, "samd_debug_replay_trace: bad arguments");
    replay_trace_kernel<<<h->a.n_requests, with_scout ? 64 : 32, 0, (cudaStream_t)stream>>>(h->a, trace_dev, cap, (long long *)cycles_dev);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
