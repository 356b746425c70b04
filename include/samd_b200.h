/*
 * samd_b200.h - C ABI of the B200-native SAM-Decoding hot path (libsamd_b200.so).
 *
 * The reference (hyx1999/SAM-Decoding) is pure Python and has no FFI of its own; the
 * boundary it exposes for this path is the Python class surface of samd/ and
 * samd_sam_only/ (SURVEY.md section 8b).  Every entry point below names the reference
 * method(s) it replaces (file:line relative to the reference checkout).  The Python
 * drop-in packages under sam-decoding_b200/{samd,samd_sam_only} bind these symbols with
 * ctypes (sam-decoding_b200/samd_b200/_cabi.py); INTEGRATION.md shows the stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; `stream` is a cudaStream_t passed as void* (NULL = default stream)
 *   - pointers named *_dev are device pointers, *_host are host pointers
 *   - every function returns 0 on success, non-zero on error (samd_last_error() explains)
 *   - no call synchronises the stream unless its comment says so
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 */
#ifndef SAMD_B200_H
#define SAMD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SAMD_ABI_VERSION 3

/* draft flavours (which reference package's rules apply) */
#define SAMD_FLAVOUR_SAMD      0   /* samd/draft.py:52-63, fixed n_predicts, zero padding      */
#define SAMD_FLAVOUR_SAM_ONLY  1   /* samd_sam_only/draft.py:49-59, n = min(max,1+int(m*alpha)) */

/* draft source written to out_type */
#define SAMD_DRAFT_DYN_SEQ     0   /* sequence read from the request's own history             */
#define SAMD_DRAFT_STATIC_SEQ  1   /* sequence read from the static corpus                     */
#define SAMD_DRAFT_TREE_MODEL  2   /* samd: match below len_threshold -> tree-model fallback   */
#define SAMD_DRAFT_STATIC_TREE 3   /* sam_only: static SAM wins -> samd_static_tree_draft      */

/* logits dtypes */
#define SAMD_DTYPE_BF16 0
#define SAMD_DTYPE_FP16 1
#define SAMD_DTYPE_FP32 2

typedef struct samd_dyn_s    *samd_dyn_t;     /* batch of per-request dynamic automata        */
typedef struct samd_static_s *samd_static_t;  /* read-only static automaton over a corpus     */
typedef struct samd_verify_s *samd_verify_t;  /* scratch of the verify+compact kernel         */

int         samd_abi_version(void);
const char *samd_last_error(void);            /* thread-local message of the last failure     */
int         samd_device_count(void);          /* 0 without a usable CUDA device               */

/* ----------------------------------------------------------------------------------------
 * Dynamic suffix automaton, one per request           (samd/sam/dyn_sam.py:8-113,
 *                                                       samd_sam_only/sam/dyn_sam.py:11-121)
 * Per-request arenas in HBM: 64-byte state records {link, length, min_endpos, five inline
 * out-edges, overflow list head/tail}, an open-addressing overflow table keyed (state, token)
 * for states with more than five out-edges (16 B slots, 128 B buckets), the token history
 * (1-based, text[0] = -1) and a small meta block.  Token ids must be non-negative.
 * -------------------------------------------------------------------------------------- */
/* DynSAM.__init__ for n_requests independent requests; max_tokens bounds prompt + decoded. */
int samd_dyn_create(int n_requests, int max_tokens, samd_dyn_t *out);
int samd_dyn_destroy(samd_dyn_t h);
/* DynSAM.reset (dyn_sam.py:27-34) for requests with mask_dev[r] != 0 (NULL = all). */
int samd_dyn_reset(samd_dyn_t h, const uint8_t *mask_dev, void *stream);
/* device bytes held by the arenas */
int64_t samd_dyn_bytes(samd_dyn_t h);
/* Snapshot / restore: copy every arena of `src` into `dst` (same n_requests, max_tokens). */
int samd_dyn_copy(samd_dyn_t dst, samd_dyn_t src, void *stream);
/* Per-request copy, for prefix reuse: the automaton of P + S is the automaton of P extended by S (the online
 * construction of dyn_sam.py:41-67 is deterministic), so a request whose prompt starts with a registered P starts from a
 * copy of P's automaton.  For each pair i, request dst_idx_dev[i] of `dst` becomes an exact copy of request
 * src_idx_dev[i] of `src`: state records, overflow table, token history and the 16 meta words (cursor included).  Both
 * handles must have the same max_tokens (equal record, overflow-table and history capacities: nothing is re-hashed).
 * The arena invariants hold afterwards: the source's live records are copied and the EMPTY TEMPLATE is written over the
 * destination's records beyond them, up to its own former n_states - the traffic follows the live sizes, plus the whole
 * overflow table.  dst_idx_dev entries must be distinct, and none may name a request of `src` that another pair writes.
 * One launch; the arguments do not depend on the step. */
int samd_dyn_clone(samd_dyn_t dst, const int32_t *dst_idx_dev, samd_dyn_t src, const int32_t *src_idx_dev,
                   int32_t n_pairs, void *stream);
/* Capacity growth: a new batch with max_tokens = new_max_tokens holding the same automata (state
 * numbering, cursors and histories preserved; the edge tables are re-hashed).  Synchronises; the
 * old handle stays valid and must still be destroyed by the caller. */
int samd_dyn_grow(samd_dyn_t old_handle, int new_max_tokens, samd_dyn_t *out);
/* Sums over requests (synchronises): out[8] = {n_states, tokens, n_edges, n_clones, transition
 * probes spent in add_tokens, probes spent in lookups, requests whose arena was full when a token arrived (grow with
 * samd_dyn_grow), requests that were handed a negative token (refused: -1 marks a free edge slot in the layout)}. */
int samd_dyn_stats(samd_dyn_t h, int64_t *out_host);
/* Every request's 16 meta words {n_states, last, max_length, cur_index, cur_length, n_edges, overflow, n_clones,
 * suffix-link hops, probes, ...} to the host (synchronises): per-request counters for profiling. */
int samd_dyn_meta(samd_dyn_t h, int32_t *meta_host);
/* Copy one request's automaton to the host (synchronises): meta[8] = {n_states, last,
 * max_length, cur_index, cur_length, n_edges, overflow, n_clones}; link/length/min_endpos
 * arrays of n_states entries (pass NULL to skip) and the token history text[0..max_length]. */
int samd_dyn_export(samd_dyn_t h, int request, int32_t *meta_host, int32_t *link_host, int32_t *length_host,
                    int32_t *endpos_host, int32_t *text_host, int64_t capacity);

/* Edges of one request as (state, token, target) triples, per state oldest-first (synchronises). */
int samd_dyn_export_edges(samd_dyn_t h, int request, int32_t *edges_host, int64_t capacity);
/* DynSAM.gen_draft for arbitrary state indices (samd/sam/dyn_sam.py:107-113 with to_anc;
 * samd_sam_only/sam/dyn_sam.py:116-121 when flavour = SAM_ONLY, which also needs match_dev). */
int samd_dyn_gen_draft(samd_dyn_t h, const int32_t *index_dev, const int32_t *match_dev, const int32_t *start_tok_dev,
                       int32_t flavour, int32_t n_predicts, double alpha, int32_t *out_draft_dev, int32_t draft_stride,
                       int32_t *out_len_dev, void *stream);

/* ----------------------------------------------------------------------------------------
 * Static suffix automaton over a corpus               (samd/sam/static_sam.py:8-137,
 *                                                       samd_sam_only/sam/static_sam.py:22-215)
 * -------------------------------------------------------------------------------------- */
/* StaticSAM.build (static_sam.py:38-46; build_sam, samd/sam/utils.py:10-18): host-side online
 * construction over doc_1 EOS doc_2 EOS ... (EOS appended unless the doc ends with it), flat
 * upload to the current device.  with_counts != 0 also computes cnt_endpos and the stable
 * top-8 successor table (samd_sam_only/sam/static_sam.py:94-96,137-146).  Synchronises. */
int samd_static_build(const int32_t *docs_flat_host, const int64_t *doc_offsets_host, int64_t n_docs, int32_t eos,
                      int with_counts, samd_static_t *out);
/* The two halves of samd_static_build: host construction only (no CUDA device needed; lets the
 * builder be checked on a CPU-only machine and its result saved), and the upload. */
int samd_static_build_host(const int32_t *docs_flat_host, const int64_t *doc_offsets_host, int64_t n_docs, int32_t eos,
                           int with_counts, samd_static_t *out);
int samd_static_upload(samd_static_t h);
/* Free the host mirrors of an uploaded automaton (they only serve export / save); queries keep working. */
int samd_static_drop_host(samd_static_t h);
int samd_static_destroy(samd_static_t h);
/* info[8] = {n_states, n_edges, n_tokens, n_slots, device_bytes, with_counts, n_clones, 0} */
int samd_static_info(samd_static_t h, int64_t *info_host);
/* Host copies for parity tests: link/length/min_endpos/cnt_endpos [n_states], topk [n_states*8*2]
 * as (token,target) pairs, -1 padded.  NULL skips an array. */
int samd_static_export(samd_static_t h, int32_t *link_host, int32_t *length_host, int32_t *endpos_host,
                       int32_t *count_host, int32_t *topk_host);
/* Converter for automata built elsewhere - the object graph of a reference pickle
 * (load_sam, samd/sam/utils.py:24-37): state arrays [n_states] (endpos_host = min_endpos for the
 * samd flavour, count_host = cnt_endpos for samd_sam_only; either may be NULL) and the edges as
 * (state, token, target) triples, per state in dict insertion order.  text_host[0..n_tokens] is the
 * 1-based token array (NULL for samd_sam_only, which keeps none).  Host only; call
 * samd_static_upload afterwards. */
int samd_static_from_arrays(int64_t n_states, const int32_t *link_host, const int32_t *length_host,
                            const int32_t *endpos_host, const int32_t *count_host, int64_t n_edges,
                            const int32_t *edges_host, int64_t n_tokens, const int32_t *text_host, samd_static_t *out);
/* The inverse: edges [n_edges][3] per state oldest-first, text [n_tokens+1].  NULL skips. */
int samd_static_export_edges(samd_static_t h, int32_t *edges_host, int32_t *text_host);
/* StaticSAM.gen_draft (samd/sam/static_sam.py:119-125) for arbitrary state indices. */
int samd_static_gen_draft(samd_static_t h, const int32_t *index_dev, const int32_t *start_tok_dev, int n_requests,
                          int32_t n_predicts, int32_t *out_draft_dev, int32_t draft_stride, void *stream);
/* dump_sam / load_sam (samd/sam/utils.py:20-37) in a flat, mmap-able format. */
int samd_static_save(samd_static_t h, const char *path);
int samd_static_load(const char *path, samd_static_t *out);
int samd_static_load_host(const char *path, samd_static_t *out);   /* no upload */
/* Pin the hottest prefix of the automaton (state records first, then the transition
 * table) in L2 through an access-policy window on `stream`; bytes <= 0 removes it. */
int samd_static_set_l2_window(samd_static_t h, void *stream, int64_t bytes);

/* ----------------------------------------------------------------------------------------
 * The per-step draft kernel: DraftModel.update + DraftModel.lookup, batched
 *   (samd/draft.py:52-79, samd_sam_only/draft.py:49-67; DynSAM.add_tokens dyn_sam.py:84-88,
 *    StaticSAM.transfer_tokens static_sam.py:102-104, lookup :106-109, gen_draft :107-125)
 * One warp per request.  Phase 1 (tokens_dev != NULL): append counts[r] tokens to request
 * r's dynamic automaton (match-then-append, clone-on-split) and advance its static cursor.
 * Phase 2 (start_tok_dev != NULL): peek both automata with the candidate next token, select
 * the draft source by match length and write the draft tokens.
 * -------------------------------------------------------------------------------------- */
typedef struct samd_step_args {
    samd_dyn_t     dyn;              /* required */
    samd_static_t  stat;             /* NULL = NullStaticSAM (samd/sam/static_sam.py:128-137) */
    int32_t       *static_cursor_dev;/* [n_requests][2] (index, length), in/out; NULL iff stat NULL */
    const int32_t *tokens_dev;       /* [n_requests][token_stride] accepted tokens, or NULL */
    int32_t        token_stride;
    const int32_t *counts_dev;       /* [n_requests] tokens to append this step (0 allowed) */
    const int32_t *start_tok_dev;    /* [n_requests] candidate next token, or NULL (no lookup) */
    int32_t        flavour;          /* SAMD_FLAVOUR_* */
    int32_t        n_predicts;       /* samd: n_predicts; sam_only: max_predicts */
    int32_t        len_bias;
    int32_t        len_threshold;    /* samd only */
    double         alpha;            /* sam_only only */
    /* outputs, each [n_requests] unless noted; any may be NULL */
    int32_t *out_type_dev;           /* SAMD_DRAFT_* */
    int32_t *out_match_dyn_dev;
    int32_t *out_match_static_dev;   /* unbiased */
    int32_t *out_index_dyn_dev;
    int32_t *out_index_static_dev;
    int32_t *out_draft_dev;          /* [n_requests][draft_stride] */
    int32_t  draft_stride;
    int32_t *out_draft_len_dev;
} samd_step_args;

int samd_step(const samd_step_args *args, void *stream);
/* Staging copy for the host-buffer path, as a kernel launch: dst[0:n_bytes] = src[0:n_bytes] with 16-byte coalesced
 * accesses.  Either side may be mapped pinned host memory (cudaHostAlloc / torch pin_memory) or device memory; both
 * pointers 16-byte aligned, n_bytes a multiple of 4.  A caller whose tokens / counts / start tokens live in pinned host
 * memory stages them with ONE such launch in front of samd_step (the reference has no counterpart: its DraftModel.update
 * takes Python lists, samd/draft.py:52-58); cheaper than a copy-engine node in the same graph and than letting every
 * request's CTA read its own few words across PCIe. */
int samd_stage_copy(void *dst, const void *src, int64_t n_bytes, void *stream);
/* profiling hook: when non-NULL, every samd_step launch that performs a lookup writes each request's SM
 * cycle counts to cycles_dev[16][n_requests].  Variant 0: whole request, cursor transfers, appends, lookup + draft, then
 * inside the appends: chain look-ups, edge inserts, (unused), target record, clone overflow copy, clone redirect walk.
 * Variant 1: whole request, cycles waiting for record loads, update phase, lookup phase, number of record loads that took
 * < 120 / < 500 / < 1100 / more cycles, overflow-probe cycles and count, then %globaltimer (ns) at the builder's start and
 * end (rows 10, 11), cycles in the cursor walks, in the clones' redirect walks and before the first token (rows 12-14), records read by the redirect walks (row 15). */
void samd_step_set_debug_cycles(int64_t *cycles_dev);
/* tuning hook: scout (prefetcher) warps of samd_step - 0 none, 1 the cursor scouts, 2 (default) also the redirect scout */
void samd_step_set_scouts(int on);
/* kernel variant of samd_step: 1 (default) = one thread per request walks, records held in its registers
 * (csrc/sam_scalar.cuh); 0 = the warp-cooperative probe of round 1.  Same results; kept for A/B measurements. */
void samd_step_set_variant(int variant);
/* tuning hook (variant 1): after a step's lookup the cursor scouts keep walking along the first n draft tokens - the path
 * the NEXT step's accepted tokens will most likely take - so that its records are in L2 by then.  0 = off. */
void samd_step_set_prewalk(int n_tokens);
/* tuning hook (variant 1): depth of the short-context scouts - one idle lane per token of the step walks from the root
 * through that token and the next `depth` ones, requesting the records and overflow slots a falling-back cursor walk ends
 * at.  -1 = off, 0 = only the root's slots, default 6. */
void samd_step_set_ngram(int depth);
/* tuning hook (variant 1): 1 = always the lean build (64 registers, two warps, 16 CTAs per SM), 0 = always the wide one
 * (three warps; 80 registers and 8 CTAs per SM without a static automaton, 88 and 6 with one), -1 (default) = lean when the
 * batch exceeds one wave of the wide build. */
void samd_step_set_lean(int mode);
/* profiling hook (variant 1): when non-NULL, every samd_step launch writes, per request, trace_dev[r][0] = the number of
 * state records its builder read and trace_dev[r][1..] = their state indices in order (capacity `cap` words per
 * request) - the request's dependent-load chain, replayed as bare loads by samd_debug_replay_trace. */
void samd_step_set_trace(int32_t *trace_dev, int cap);

/* Cursor-only walks.  samd_static_walk = StaticSAM.transfer_tokens (static_sam.py:102-104) when
 * tokens_dev != NULL, then StaticSAM.lookup (:106-109) when peek_tok_dev != NULL (non-mutating).
 * samd_dyn_transfer = DynSAM.transfer_tokens (dyn_sam.py:90-92): moves the cursor, appends nothing. */
int samd_static_walk(samd_static_t h, int32_t *static_cursor_dev, const int32_t *tokens_dev, int32_t token_stride,
                     const int32_t *counts_dev, const int32_t *peek_tok_dev, int n_requests, int32_t *out_index_dev,
                     int32_t *out_len_dev, void *stream);
int samd_dyn_transfer(samd_dyn_t h, const int32_t *tokens_dev, int32_t token_stride, const int32_t *counts_dev, void *stream);

/* sam_only static tree drafter (samd_sam_only/sam/static_sam.py:148-215): best-first search
 * over occurrence-count ratios with CPython-heapq tie order, for the requests whose
 * type_dev[r] == SAMD_DRAFT_STATIC_TREE (type_dev NULL = all).  Writes per request the tree
 * tokens and parent indices [max_nodes], the node count, the per-node depth
 * (= tree_position_ids), and the padded retrieve table [max_paths][max_depth] (-1 padded,
 * leaves ascending) with its shape.  match_static_dev is the UNBIASED match length. */
int samd_static_tree_draft(samd_static_t h, int n_requests, const int32_t *type_dev, const int32_t *index_static_dev,
                           const int32_t *match_static_dev, const int32_t *start_tok_dev, int32_t max_predicts,
                           double alpha, int32_t K, int32_t len_bias, int32_t *out_tokens_dev,
                           int32_t *out_parents_dev, int32_t *out_depth_dev, int32_t *out_n_nodes_dev,
                           int32_t *out_retrieve_dev, int32_t max_paths, int32_t max_depth,
                           int32_t *out_retrieve_shape_dev, void *stream);

/* sam_only batch buffers (gen_buffers samd_sam_only/sam/static_sam.py:148-180, sequence positions
 * samd_sam_only/sam/dyn_sam.py:116-121, the mask splice samd_sam_only/model_patch/llama.py:94-96, the decode step
 * samd_sam_only/samd_model.py:117-157): per request b, its sequence draft (samd_step: draft_len tokens) or, when
 * type_dev[b] == SAMD_DRAFT_STATIC_TREE, its static tree (samd_static_tree_draft) becomes uniform rows:
 *   tokens[b][T]            node tokens, 0 past the request's node count
 *   position_ids[b][T]      cache_len[b] + depth of the node (a sequence: the node index; pad rows: the row index)
 *   n_nodes[b], n_paths[b]
 *   retrieve[b][P][D]       a tree's leaf paths, or the sequence's one path 0..draft_len-1; -1 padded
 *   mask[b][T][kv_len]      additive, in the LM's dtype: 0 where node i may attend, the dtype's lowest finite value
 *                           (torch.finfo(dtype).min) elsewhere.  Node i sees every column < cache_len[b] and column
 *                           cache_len[b] + j for j = i and every ancestor of i (a sequence: every j <= i).  Rows
 *                           i >= n_nodes[b] see the past and themselves, never nothing.
 * Any type other than SAMD_DRAFT_STATIC_TREE is a sequence, and a non-tree request's tree arrays are not read (they are
 * stale).  tree_tokens_dev NULL = no tree drafter: every request is a sequence.  A finished request (done_dev[b] != 0)
 * gets a one-node draft: n_nodes = 1, retrieve row 0 = [0, -1, ...], n_paths = 0 - the verify walk accepts nothing and
 * maps index 0 to 0, so samd_verify_compact moves none of its KV rows.  T <= 256, kv_len >= T.  No argument depends on
 * the step, so the launch can be captured in a CUDA graph. */
typedef struct samd_assemble_args {
    int32_t        batch;
    int32_t        n_nodes;           /* T: node rows per request */
    int32_t        n_paths, depth;    /* P x D path table */
    const int32_t *type_dev;          /* [B] SAMD_DRAFT_* (samd_step out_type), or NULL = all sequences */
    const int32_t *draft_dev;         /* [B][draft_stride] sequence drafts (samd_step out_draft) */
    int32_t        draft_stride;
    const int32_t *draft_len_dev;     /* [B] */
    /* samd_static_tree_draft outputs, or tree_tokens_dev NULL */
    const int32_t *tree_tokens_dev, *tree_parents_dev, *tree_depth_dev;  /* [B][tree_stride], tree_stride <= T */
    int32_t        tree_stride;
    const int32_t *tree_n_dev;        /* [B] */
    const int32_t *tree_retrieve_dev; /* [B][tree_max_paths][tree_max_depth], tree_max_paths <= P, tree_max_depth <= D */
    int32_t        tree_max_paths, tree_max_depth;
    const int32_t *tree_shape_dev;    /* [B][2] {leaves, deepest path} */
    const int32_t *cache_len_dev;     /* [B] */
    const uint8_t *done_dev;          /* [B] finished requests, or NULL */
    int32_t        mask_dtype;        /* SAMD_DTYPE_* */
    int32_t        kv_len;
    /* outputs */
    int32_t *out_tokens_dev;          /* [B][T] */
    int64_t *out_position_ids_dev;    /* [B][T] */
    int32_t *out_n_nodes_dev, *out_n_paths_dev;   /* [B] */
    int32_t *out_retrieve_dev;        /* [B][P][D] */
    void    *out_mask_dev;            /* [B][T][kv_len] */
} samd_assemble_args;
int samd_draft_assemble(const samd_assemble_args *args, void *stream);

/* ----------------------------------------------------------------------------------------
 * Document-sharded static SAM (SURVEY.md section 8e): per-shard packed keys
 *   key = (match_len << 32) | (0xFFFFFFFF - (shard_offset + min_endpos)), 0 when no match,
 * to be max-reduced across shards (ncclMax on 64-bit), then the draft is read from the
 * replicated corpus token array at the winning global position.
 * -------------------------------------------------------------------------------------- */
int samd_static_lookup_keys(samd_static_t h, const int32_t *static_cursor_dev, const int32_t *start_tok_dev,
                            int n_requests, int64_t shard_offset, int64_t *out_keys_dev, void *stream);
int samd_draft_from_keys(const int64_t *keys_dev, const int32_t *corpus_dev, int64_t n_corpus_tokens,
                         const int32_t *start_tok_dev, int n_requests, int32_t n_predicts, int32_t *out_match_dev,
                         int32_t *out_draft_dev, int32_t draft_stride, void *stream);

/* The same reduction without a collective library (one process per GPU, NVLink peer memory): every rank owns an
 * exchange buffer, maps every peer's through CUDA IPC, and the look-up kernel itself max-reduces the packed keys into
 * EVERY rank's buffer with remote atomics; the draft kernel waits for all shards' keys on the local buffer.
 *   samd_xchg_create           this rank's buffer for n_queries queries (cudaMalloc)
 *   samd_xchg_export           its 64-byte CUDA IPC handle, to be all-gathered by the caller (torch.distributed)
 *   samd_xchg_connect          handles = [world][64] in rank order; opens the peers' buffers
 *   samd_static_lookup_exchange / samd_draft_from_exchange   replace samd_static_lookup_keys + all-reduce-max +
 *                              samd_draft_from_keys; every rank must issue the same sequence of pairs.  No argument
 *                              depends on the step, so the pair can be captured in a CUDA graph. */
typedef struct samd_xchg_s *samd_xchg_t;
int samd_xchg_create(int rank, int world, int n_queries, samd_xchg_t *out);
int samd_xchg_export(samd_xchg_t x, void *handle64_out);
int samd_xchg_connect(samd_xchg_t x, const void *handles);
int samd_xchg_destroy(samd_xchg_t x);
int samd_xchg_status(samd_xchg_t x);   /* 0 ok; 1 = a draft kernel gave up waiting for a peer after 5 s (synchronises) */
int samd_static_lookup_exchange(samd_static_t h, int32_t *static_cursor_dev, const int32_t *tokens_dev, int32_t token_stride,
                                const int32_t *counts_dev, const int32_t *start_tok_dev, int64_t shard_offset, samd_xchg_t x,
                                void *stream);   /* tokens_dev != NULL: StaticSAM.transfer_tokens first, same launch */
int samd_draft_from_exchange(samd_xchg_t x, const int32_t *corpus_dev, int64_t n_corpus_tokens, const int32_t *start_tok_dev,
                             int32_t n_predicts, int32_t *out_match_dev, int32_t *out_draft_dev, int32_t draft_stride,
                             void *stream);

/* ----------------------------------------------------------------------------------------
 * Fused greedy verification + KV-cache compaction
 *   (gather samd/samd_model.py:159-168, eval_posterior greedy samd/utils.py:127-141,
 *    update_state samd/samd_model.py:185-211, SamdStaticCache.select_indices samd/cache.py:118-133)
 * One persistent launch: streams logits [B,T,V] once (row argmax with torch.argmax's
 * lowest-index / NaN-is-max rule), walks the P x D path table per request, writes best /
 * accept_len (= accepted + 1) / next_token / accepted tokens + indices, then moves KV rows
 * cache_len+indices[j] -> cache_len+j in every K and V tensor and bumps cache_len.
 * -------------------------------------------------------------------------------------- */
int samd_verify_create(int max_batch, int max_nodes, samd_verify_t *out);
int samd_verify_destroy(samd_verify_t h);

typedef struct samd_verify_args {
    const void    *logits_dev;        /* [B][T][V], dtype below */
    int32_t        dtype;             /* SAMD_DTYPE_* */
    int32_t        batch, n_nodes, vocab;
    int64_t        batch_stride, row_stride;       /* in elements */
    const int32_t *tree_tokens_dev;   /* [B][n_nodes] draft tokens fed to the LM */
    const int32_t *n_nodes_dev;       /* [B] live rows per request, or NULL (= n_nodes) */
    const int32_t *retrieve_dev;      /* [P][D] shared, or [B][P][D] when retrieve_batch_stride != 0;
                                         NULL = one identity path of n_nodes entries (sequence) */
    int32_t        n_paths, depth;
    int64_t        retrieve_batch_stride;          /* elements; 0 = shared */
    const int32_t *n_paths_dev;       /* [B] live paths per request, or NULL */
    /* KV cache: n_kv tensors [B][H][max_len][Dh]; NULL kv_ptrs_dev or move_kv == 0 = no row moves */
    void *const   *kv_ptrs_dev;       /* device array of n_kv base pointers */
    int32_t        n_kv, n_heads, row_bytes;       /* row_bytes = Dh * sizeof(element) */
    int64_t        kv_batch_stride, kv_head_stride, kv_pos_stride;   /* bytes */
    int32_t        move_kv;
    int32_t       *cache_len_dev;     /* [B] in/out, or NULL */
    /* outputs */
    int32_t *out_best_dev, *out_accept_len_dev, *out_next_token_dev;   /* [B] */
    int32_t *out_tokens_dev, *out_indices_dev;      /* [B][depth] (sequence: [B][n_nodes]) */
    int32_t *out_node_argmax_dev;     /* [B][n_nodes] or NULL */
    /* Token Recycle (samd/tree_model/token_recycle/token_recycle.py:36-47), fused into the same pass over the logits:
     * out_topk_dev != NULL -> the 8 largest logits of every row, as indices ordered (value descending, index
     * ascending; NaN largest; column 0 = the row argmax), -1 rows for dead nodes.  recycle_table_dev != NULL ->
     * additionally table[tree_tokens[b][t]][0..7] = that row's list, the last (b, t) winning when a token feeds
     * several rows (the reference's zip order); recycle_owner_dev is [vocab] scratch holding -1 between launches. */
    int32_t *out_topk_dev;            /* [B][n_nodes][8] or NULL */
    int32_t *recycle_table_dev;       /* [vocab][8], rows of -1 = no entry; or NULL */
    int32_t *recycle_owner_dev;       /* [vocab] */
} samd_verify_args;

int samd_verify_compact(samd_verify_t h, const samd_verify_args *args, void *stream);
/* ----------------------------------------------------------------------------------------
 * Stochastic (typical-acceptance) verification: the sampling branch of eval_posterior (samd/utils.py:142-184) and the
 * draw of the token that follows (gen_candidates, samd/utils.py:85-88, torch.multinomial(sample_p, 1)), for a batch.
 * Level by level, each distinct candidate token x among the paths that share the accepted prefix is tested once, in
 * path order, with one uniform draw r:  accept iff r <= p(x) / (1 - mass rejected so far at this level), where
 * p = softmax(logits_processor(row)) and logits_processor = temperature, then top-p, then top-k (samd/utils.py:44-58).
 * Top-p follows an ascending sort that keeps equal values in index order: of the tie group the cut falls into, the
 * lowest-index members are removed while the cumulative mass stays within 1 - top_p (masses summed in double).
 * The next token is drawn from the level's residual distribution when its last level rejected something (and the path
 * is not complete), else from the plain softmax of the last accepted node's row (samd/utils.py:173-179).
 * RNG CONTRACT: Philox4x32-10; uniform number k of request b is
 *     u = (philox(counter = {lo32(c), hi32(c), 0, 0}, key = {lo32(seed_b), hi32(seed_b)})[0] >> 8) * 2^-24,  c = offset_b + k
 * one draw per tested candidate, then one for the next token (inverse CDF in token-id order); offsets_dev[b] is advanced
 * by the draws used, so consecutive calls continue one stream per request.  Python's random.random() of the reference
 * cannot be reproduced bit for bit: decisions are exact against the oracle given the same stream
 * (tests/test_gpu_sampling.py) and the acceptance-length / next-token statistics match the reference's own function.
 * -------------------------------------------------------------------------------------- */
typedef struct samd_sample_args {
    const void    *logits_dev;        /* [B][T][V], dtype below */
    int32_t        dtype;             /* SAMD_DTYPE_* */
    int32_t        batch, n_nodes, vocab;
    int64_t        batch_stride, row_stride;       /* in elements */
    const int32_t *tree_tokens_dev;   /* [B][n_nodes] */
    const int32_t *retrieve_dev;      /* [P][D] shared, or [B][P][D] when retrieve_batch_stride != 0; NULL = one identity path */
    int32_t        n_paths, depth;
    int64_t        retrieve_batch_stride;
    const int32_t *n_paths_dev;       /* [B] live paths per request (<= n_paths), or NULL */
    float          temperature;       /* >= 1e-5 */
    float          top_p;             /* active when 1e-8 <= top_p < 1 */
    int32_t        top_k;             /* active when > 0 */
    const uint64_t *seeds_dev;        /* [B] */
    uint64_t      *offsets_dev;       /* [B] in/out */
    int32_t *out_best_dev, *out_accept_len_dev, *out_next_token_dev;   /* [B]; accept_len = accepted + 1 */
    int32_t *out_tokens_dev, *out_indices_dev;      /* [B][depth] (identity path: [B][n_nodes]); -1 past accept_len */
    float   *out_sample_p_dev;        /* [B][V] the next token's distribution (the reference's returned sample_p), or NULL */
} samd_sample_args;
int samd_verify_sample(const samd_sample_args *args, void *stream);
/* The same launch with per-request arguments (every pointer NULL = the shared value of `args`), for a batch whose
 * requests each have their own processor, path-table width and state - what a batched decoder with per-request
 * sampling parameters needs.  Per request b:
 *   temperature / top_p / top_k   its own processor (same validity rules as the scalars; not checked on the host)
 *   greedy_dev[b] = 1             the greedy eval_posterior (samd/utils.py:127-141) instead of the typical walk: the
 *                                 argmax of every node row (torch.argmax's rule), the match length of every path, the
 *                                 first longest path, the next token = the argmax of its last accepted row; no draw -
 *                                 the outputs equal samd_verify_compact's for the same rows and table
 *   done_dev[b] = 1, or n_paths 0 a finished request: no draw, offsets_dev[b] untouched, accept_len 0 and no other output
 *                                 (samd_kv_compact then moves none of its rows)
 *   n_nodes_dev[b]                its own row count: a -1 entry of its paths wraps to row n_nodes_dev[b] - 1
 *   depth_dev[b]                  its own path width (<= depth): the walk stops there, so -1 pads beyond a request's
 *                                 own draft are never compared (inside it, a -1 selects token 0 as in the reference)
 * The output layout is samd_verify_sample's ([B][depth] tokens / indices).  Greedy requests need n_nodes <= 256.  No
 * argument depends on the step, so the launch can be captured in a CUDA graph. */
typedef struct samd_sample_request_args {
    const float   *temperature_dev;   /* [B]; NULL = args->temperature */
    const float   *top_p_dev;         /* [B]; NULL = args->top_p */
    const int32_t *top_k_dev;         /* [B]; NULL = args->top_k */
    const uint8_t *greedy_dev;        /* [B] 1 = greedy eval_posterior for this request; NULL = none */
    const uint8_t *done_dev;          /* [B] 1 = finished slot: no draw, no output but accept_len 0; NULL = none */
    const int32_t *n_nodes_dev;       /* [B] the request's own node count (-1 wraps to ITS last row); NULL = n_nodes */
    const int32_t *depth_dev;         /* [B] the request's own path width; NULL = depth */
} samd_sample_request_args;
int samd_verify_sample_requests(const samd_sample_args *args, const samd_sample_request_args *r, void *stream);

/* Per-token log-probabilities of the accepted path of every request, from the logits a verify launch read.  For request
 * b with a = min(count_dev[b], width) >= 1 and not done, position j < a is scored on row r = indices_dev[b][j] (NULL
 * indices: r = j; a -1 entry: the request's last live row n_nodes_dev[b] - 1, as samd_verify_compact reads it) against
 * the target tokens_dev[b][j + 1] when j + 1 < a, else next_token_dev[b]:
 *     logprob = log_softmax(float32(row))[target]      (raw: no temperature, top-p or top-k)
 * and, with n_top > 0, the n_top largest entries of the row (value descending, index ascending, NaN largest) with their
 * log-probabilities.  Positions j < a - 1 go to out_logprob_dev[b][j] / out_top_*[b][j][:], the last one to
 * out_next_logprob_dev[b] / out_next_top_*[b][:].  A -inf logit gives -inf, a row with a NaN gives NaN, a target
 * outside [0, V) gives NaN.  Requests with a = 0 or done write nothing, nor does any position j >= a.  Only the scored
 * rows are read, each once.  The reduction order depends only on V and the launch shape, so a row gives bit-identical
 * results wherever it sits; no argument depends on the step, so the launch can be captured in a CUDA graph. */
typedef struct samd_logprob_args {
    const void    *logits_dev;        /* [B][n_nodes][V], dtype below */
    int32_t        dtype;             /* SAMD_DTYPE_* */
    int32_t        batch, n_nodes, vocab;
    int64_t        batch_stride, row_stride;       /* in elements */
    const int32_t *indices_dev;       /* [B][width] path row indices (a verify launch's out_indices), or NULL = identity */
    int32_t        width;             /* row length of indices_dev, tokens_dev and out_logprob_dev (<= n_nodes if identity) */
    const int32_t *count_dev;         /* [B] scored positions (a verify launch's accept_len) */
    const int32_t *tokens_dev;        /* [B][width] path tokens (out_tokens); may be NULL when every count is <= 1 */
    const int32_t *next_token_dev;    /* [B] */
    const int32_t *n_nodes_dev;       /* [B] live rows per request, or NULL = n_nodes */
    const uint8_t *done_dev;          /* [B] 1 = finished: nothing written, or NULL */
    int32_t        n_top;             /* 0 .. 8 */
    float   *out_logprob_dev;         /* [B][width] (only NULL when width == 1) */
    float   *out_next_logprob_dev;    /* [B] */
    int32_t *out_top_ids_dev;         /* [B][width][n_top] (n_top > 0) */
    float   *out_top_logprob_dev;     /* [B][width][n_top] */
    int32_t *out_next_top_ids_dev;    /* [B][n_top] */
    float   *out_next_top_logprob_dev;/* [B][n_top] */
} samd_logprob_args;
int samd_token_logprobs(const samd_logprob_args *args, void *stream);

/* Repetition, presence and frequency penalties on the draft rows of a batch, in place, before a verify launch reads them
 * (HF RepetitionPenaltyLogitsProcessor; presence / frequency as in the OpenAI API).  Row j < n_nodes_dev[b] of row-batch
 * b belongs to state row s = slots_dev[b] (NULL: s = b); its context is the prompt, the emitted tokens and the node tokens
 * on the path from node 0 to node j, both included (NULL tokens_dev: no draft context, e.g. the prompt's last row).  With
 * c[t] = the output count counts_dev[s][t] & 0x7FFFFFFF plus the occurrences of t on that path, and seen[t] = bit 31 of
 * counts_dev[s][t] (t is in the prompt) or c[t] > 0, every seen entry becomes, in fp32, each operation rounded on its own:
 *     x = x < 0 ? x * r : x / r;   x = x - f * (float)c[t];   x = x - p * (c[t] > 0 ? 1 : 0)
 * and is rounded to nearest into the logits dtype (-inf stays -inf, NaN stays NaN).  Untouched: unseen entries, requests
 * with r = 1 and p = f = 0, done requests, rows at or past n_nodes_dev[b], and, with a path table, rows on none of the
 * request's first n_paths_dev[b] paths (a path ends at its first -1).  Each entry is rewritten at most once, from its own
 * inputs, so the results do not depend on the launch shape; no argument depends on the step, so the launch can be
 * captured in a CUDA graph. */
typedef struct samd_penalty_args {
    void          *logits_dev;        /* [B][n_nodes][V], dtype below, rewritten in place */
    int32_t        dtype;             /* SAMD_DTYPE_* */
    int32_t        batch, n_nodes, vocab;          /* n_nodes <= 256 */
    int64_t        batch_stride, row_stride;       /* in elements */
    const int32_t *tokens_dev;        /* [B][n_nodes] node tokens, or NULL = no row has draft context */
    const int32_t *retrieve_dev;      /* [B][n_paths][depth] path table, -1 padded, or NULL = the identity chain */
    int32_t        n_paths, depth;
    const int32_t *n_nodes_dev;       /* [B] live rows per request, or NULL = n_nodes */
    const int32_t *n_paths_dev;       /* [B] live paths per request, or NULL = n_paths */
    const uint8_t *done_dev;          /* [B] 1 = finished: not touched, or NULL */
    const int32_t *slots_dev;         /* [B] state row of each row-batch entry, or NULL = identity */
    int32_t        n_slots;           /* S */
    const int32_t *counts_dev;        /* [S][V] output count (bits 0..30) | seen in the prompt (bit 31) */
    const float   *repetition_dev;    /* [S] r > 0 */
    const float   *presence_dev;      /* [S] p */
    const float   *frequency_dev;     /* [S] f */
} samd_penalty_args;
int samd_apply_penalties(const samd_penalty_args *args, void *stream);

/* Stop sequences: where does this step's output end?  Request b has emitted hist_dev[b][0 .. hist_len_dev[b]) so far
 * and this step would emit tokens_dev[b][0 .. count_dev[b]).  Sequence j (stop_len_dev[b][j] = L in [1, 16] ids
 * stop_tokens_dev[b][j][0 .. L); L = 0 marks an unused entry) ends at step position i < count when the output tokens
 * at output positions hist_len + i - L + 1 .. hist_len + i equal it; positions before 0 (the prompt) never match, and
 * only the last SAMD_STOP_MAX_LEN - 1 history tokens are read.  out_count_dev[b] = e + 1 for the earliest such i = e,
 * out_hit_dev[b] = the lowest j ending there; without a match, or for a done request or count 0: count and -1.  Tokens
 * at or past count are never read.  out_count_dev may alias count_dev.  The result depends only on the inputs; no
 * argument depends on the step, so the launch can be captured in a CUDA graph. */
#define SAMD_STOP_MAX_SEQS 16
#define SAMD_STOP_MAX_LEN  16
typedef struct samd_stop_args {
    int32_t        batch, width;      /* width <= 256 */
    const int32_t *tokens_dev;        /* [B][width] this step's accepted tokens */
    const int32_t *count_dev;         /* [B] candidate tokens (<= width) */
    const int32_t *hist_dev;          /* [B][hist_stride] output emitted so far */
    int32_t        hist_stride;
    const int32_t *hist_len_dev;      /* [B] */
    const int32_t *stop_tokens_dev;   /* [B][SAMD_STOP_MAX_SEQS][SAMD_STOP_MAX_LEN] */
    const int32_t *stop_len_dev;      /* [B][SAMD_STOP_MAX_SEQS], 0 = unused */
    const uint8_t *done_dev;          /* [B] 1 = finished, or NULL */
    int32_t       *out_count_dev;     /* [B] */
    int32_t       *out_hit_dev;       /* [B] sequence index or -1 */
} samd_stop_args;
int samd_stop_match(const samd_stop_args *args, void *stream);

/* Logit bias, banned token sequences and min_tokens on the draft rows of a batch, in place, after any penalties and
 * before a verify launch reads them.  Row j < n_nodes_dev[b] of row-batch b belongs to state row s = slots_dev[b] (NULL:
 * s = b).  Its context is the output so far, hist_dev[s][0 .. hist_len_dev[s]) (NULL hist_len_dev: empty), then the node
 * tokens on the path from node 0 to node j, both included; node 0 sits at output position hist_len, so a node at depth d
 * predicts output position hist_len + d + 1.  NULL tokens_dev is the admission form: no node tokens, every row predicts
 * position hist_len.  In this order:
 *   - bias: for each of the slot's bias_n_dev[s] entries (distinct ids), x = round_to_dtype(fp32(x) + bias); a -inf bias
 *     stores -inf (a ban, whatever x was).  -inf stays -inf and NaN stays NaN under a finite bias.
 *   - bans, each storing -inf: for every bad word (bad_len_dev[s][k] = L in [1, 16]; 0 = unused) whose first L - 1 ids
 *     end the row's context, its last id (L = 1: banned on every row); and on a row predicting a position below
 *     min_tokens_dev[s], eos_token (>= 0) and, for every stop sequence whose first L - 1 ids end the context, its last id.
 * The context never reaches before output position 0, and only its last SAMD_BAD_MAX_LEN - 1 tokens are read.
 * Untouched: done requests, slots with no bias, no bad word and min_tokens 0, rows at or past n_nodes_dev[b], and, with a
 * path table, rows on none of the request's first n_paths_dev[b] paths (a path ends at its first -1).  Every (row, token)
 * is read-modify-written at most once; the results depend only on the inputs and no argument depends on the step, so the
 * launch can be captured in a CUDA graph. */
#define SAMD_BIAS_MAX     256
#define SAMD_BAD_MAX_SEQS 16
#define SAMD_BAD_MAX_LEN  16
typedef struct samd_logit_control_args {
    void          *logits_dev;        /* [B][n_nodes][V], dtype below, rewritten in place */
    int32_t        dtype;             /* SAMD_DTYPE_* */
    int32_t        batch, n_nodes, vocab;          /* n_nodes <= 256 */
    int64_t        batch_stride, row_stride;       /* in elements */
    const int32_t *tokens_dev;        /* [B][n_nodes] node tokens, or NULL = the admission form */
    const int32_t *retrieve_dev;      /* [B][n_paths][depth] path table, -1 padded, or NULL = the identity chain */
    int32_t        n_paths, depth;
    const int32_t *n_nodes_dev;       /* [B] live rows per request, or NULL = n_nodes */
    const int32_t *n_paths_dev;       /* [B] live paths per request, or NULL = n_paths */
    const uint8_t *done_dev;          /* [B] 1 = finished: not touched, or NULL */
    const int32_t *slots_dev;         /* [B] state row of each row-batch entry, or NULL = identity */
    int32_t        n_slots;           /* S */
    const int32_t *hist_dev;          /* [S][hist_stride] output emitted so far (may be NULL without hist_len_dev) */
    int32_t        hist_stride;
    const int32_t *hist_len_dev;      /* [S], or NULL = 0 */
    const int32_t *bias_ids_dev;      /* [S][SAMD_BIAS_MAX] distinct token ids */
    const float   *bias_dev;          /* [S][SAMD_BIAS_MAX] finite or -inf */
    const int32_t *bias_n_dev;        /* [S] entries in use */
    const int32_t *bad_tokens_dev;    /* [S][SAMD_BAD_MAX_SEQS][SAMD_BAD_MAX_LEN] */
    const int32_t *bad_len_dev;       /* [S][SAMD_BAD_MAX_SEQS], 0 = unused */
    const int32_t *min_tokens_dev;    /* [S] */
    const int32_t *stop_tokens_dev;   /* [S][SAMD_STOP_MAX_SEQS][SAMD_STOP_MAX_LEN], or NULL = no stop sequences */
    const int32_t *stop_len_dev;      /* [S][SAMD_STOP_MAX_SEQS], 0 = unused (NULL with stop_tokens_dev) */
    int32_t        eos_token;         /* -1 = none */
} samd_logit_control_args;
int samd_apply_logit_controls(const samd_logit_control_args *args, void *stream);

/* TokenRecycle.gen_draft (token_recycle.py:49-59) for a batch: tokens[b][0] = start_tok[b]; every other node takes
 * table[token of its parent][its rank among the parent's children], or 0 when the parent's token has no entry.
 * parent / rank: [n_nodes] device arrays describing the static tree (node 0 = root, parents before children);
 * type_dev != NULL restricts the fill to requests whose type equals `only_type` (others are left untouched). */
int samd_recycle_gen_tree(const int32_t *table_dev, int32_t vocab, const int32_t *parent_dev, const int32_t *rank_dev,
                          int32_t n_nodes, const int32_t *start_tok_dev, const int32_t *type_dev, int32_t only_type,
                          int32_t batch, int32_t *out_tokens_dev, void *stream);
/* tuning hook: 1 = overlapped flow of samd_verify_compact - a request is walked by the warp that reports its
 * last logits chunk and its KV rows are moved by warps that have run out of logits, while the rest still streams; no
 * grid-wide barrier.  2 = walks as requests complete + L2 prefetch of their source rows, row moves after the last walk;
 * 3 = the same without the prefetch.  0 (default) = the two-barrier flow (stream, barrier, walks, barrier, row moves):
 * measured on c4, 79.6 us against 94.7 / 152 / 82.3 for modes 1 / 2 / 3 (DESIGN.md 3.2).  Launches that also compute the
 * top-8 lists always use the barrier flow. */
void samd_verify_set_overlap(int on);
/* tuning hook: 1 (default) = only as many warps stream logits as divide the work items evenly (the rest of the grid joins
 * for the row moves); 0 = every resident warp takes items (round 1). */
void samd_verify_set_even_items(int on);
/* tuning hook: 1 = 16-bit logits are streamed through shared memory by the bulk-copy engine (cp.async.bulk + mbarrier
 * ring, 8 KB in flight per warp; UBLKCP / SYNCS in SASS); 0 (default) = register-staged 128-bit loads.  Measured on c4:
 * 56.9 vs 50.0 us verify-only (the ring's shared memory costs a quarter of the resident warps and the stream was already at
 * 6.1-7 TB/s), so the register path stays the default. */
void samd_verify_set_tma(int on);
/* tuning hook: logits elements per phase-1 work item (0 = default) */
void samd_verify_set_chunk(int elements);
/* profiling hook: [grid warps][3] uint64 globaltimer ns per warp of the next launches - start, end of the logits
 * stream, exit; NULL = off */
void samd_verify_set_debug_times(uint64_t *times_dev);
/* Stand-alone SamdStaticCache.select_indices (samd/cache.py:118-133): rows cache_len+indices[b][j] ->
 * cache_len+j for j < accept_len[b] in every KV tensor, then cache_len[b] += accept_len[b].
 * indices_dev NULL = sequence draft (only the length bump, cache.py:123-126,133). */
int samd_kv_compact(void *const *kv_ptrs_dev, int32_t n_kv, int32_t n_heads, int32_t row_bytes, int64_t kv_batch_stride,
                    int64_t kv_head_stride, int64_t kv_pos_stride, const int32_t *indices_dev, int32_t depth,
                    const int32_t *accept_len_dev, int32_t *cache_len_dev, int32_t batch, void *stream);
/* Prefix reuse at admission (the prefill a causal LM would repeat: KV row i depends only on tokens 0..i; the rows that
 * samd/cache.py:SamdStaticCache holds for one request): for each pair i, rows [0, n_rows_dev[i]) of batch row
 * src_row_dev[i] of the source cache are copied into batch row dst_row_dev[i] of the destination, in every one of the n_kv
 * tensors and every head.  Each side is described like samd_kv_compact's KV (a device table of n_kv base pointers, byte
 * strides), with its own strides: the two caches may differ in batch size and length.  n_rows 0 is allowed; nothing
 * outside the listed rows is written.  16-byte accesses where row_bytes and the alignment allow, narrower ones
 * otherwise.  One launch; the arguments do not depend on the step. */
int samd_kv_copy_rows(void *const *dst_ptrs_dev, int64_t dst_batch_stride, int64_t dst_head_stride, int64_t dst_pos_stride,
                      void *const *src_ptrs_dev, int64_t src_batch_stride, int64_t src_head_stride, int64_t src_pos_stride,
                      int32_t n_kv, int32_t n_heads, int32_t row_bytes, const int32_t *dst_row_dev,
                      const int32_t *src_row_dev, const int32_t *n_rows_dev, int32_t n_pairs, void *stream);
/* profiling aid: n_warps warps each chase `hops` dependent pointers through n_records 64-byte records
 * (record word 0 = next index); measures dependent-load latency at the step kernel's concurrency */
int samd_debug_pointer_chase(const void *recs_dev, int64_t n_records, int n_warps, int hops, int32_t *sink_dev, void *stream);
/* profiling aid: the ceiling of scattered row moves - n_granules copies of granule_bytes (a multiple of 16) each,
 * base + src_off[g] -> base + dst_off[g] (byte offsets, 16-byte aligned), four independent 16-byte units in flight per
 * lane over n_blocks x 256 threads; what samd_verify_compact's KV compaction (one 256-byte granule per tensor, head
 * and accepted row) can reach at best.  tools/row_move_ceiling.py */
int samd_debug_granule_copy(void *base_dev, const int64_t *src_off_dev, const int64_t *dst_off_dev, int64_t n_granules,
                            int32_t granule_bytes, int32_t n_blocks, void *stream);
/* profiling aid: every warp of an n_blocks x threads launch records {%smid, %warpid} into out_dev[warp][2] and lingers
 * spin_ns so that the grid is resident together - which scheduler partition (slot mod 4) the builder warps of a
 * step-shaped launch land on.  tools/warp_slots.py */
int samd_debug_warp_slots(int32_t *out_dev, int n_blocks, int threads, int spin_ns, void *stream);
/* profiling aid: the floor of samd_step's dependent-load chain.  One thread per request of `h` reads the records listed
 * in trace_dev (layout of samd_step_set_trace) one after the other, every address depending on the previous load's
 * value; with_scout != 0 adds a second thread per request that runs ahead through the same list with independent
 * loads (an ideal prefetcher).  cycles_dev[3][n_requests] = SM cycles of request r's chain, %globaltimer at its start / end. */
int samd_debug_replay_trace(samd_dyn_t h, const int32_t *trace_dev, int cap, int with_scout, int64_t *cycles_dev, void *stream);
/* number of kernel launches the library has issued (for bench.py's gpu_launches) */
int64_t samd_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SAMD_B200_H */
