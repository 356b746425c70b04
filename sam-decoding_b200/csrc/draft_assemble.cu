// Batch buffer assembly for the sam_only flavour: per request, "a sequence of draft_len tokens" (samd_step) or "a tree of
// tree_n nodes" (samd_static_tree_draft) becomes the uniform rows the LM forward and samd_verify_compact take - node
// tokens, position ids, the additive [T][kv_len] attention mask, the [P][D] path table, node and path counts.
//
// Replaces, per step and per request, what the reference does on the host:
//   gen_buffers                 samd_sam_only/sam/static_sam.py:148-180 (tree mask, depths, leaf paths)
//   sequence positions          samd_sam_only/sam/dyn_sam.py:116-121
//   the mask splice             samd_sam_only/model_patch/llama.py:94-96 (past columns + the tree block)
//   the decode step's buffers   samd_sam_only/samd_model.py:117-157
//
// One CTA per (request, tile of ASM_ROWS node rows), one warp per row.  A tree tile first builds the ancestor sets of the
// nodes it needs as bit words in shared memory: parents precede children (the drafter's numbering), so a node's set is its
// parent's set plus itself.  Then every warp streams its row of the mask with 16-byte stores; the CTA of tile 0 also
// writes the request's small outputs.  Nothing depends on the host between steps: capturable in a graph.
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#define ASM_MAX_T 256
#define ASM_WORDS (ASM_MAX_T / 32)
#define ASM_ROWS 8                       // rows per CTA = warps per CTA
#define ASM_THREADS (32 * ASM_ROWS)

struct AsmParams {
    int B, T, P, D, kv_len;
    const int32_t *type, *draft, *draft_len;
    int draft_stride;
    const int32_t *tree_tok, *tree_par, *tree_dep, *tree_n, *tree_ret, *tree_shape;
    int tree_stride, tree_paths, tree_depth;
    const int32_t *cache_len;
    const uint8_t *done;
    int32_t *tokens, *n_nodes, *n_paths, *retrieve;
    long long *pos;
    void *mask;
};

// the mask's element bits: 0 = attend, the dtype's lowest finite value (torch.finfo(dtype).min) = masked
template <int ES> struct MaskBits;
template <> struct MaskBits<2> { typedef uint16_t T; };
template <> struct MaskBits<4> { typedef uint32_t T; };

// allowed column bits of one row, word w: j <= i (sequence: the chain)
__device__ __forceinline__ uint32_t prefix_word(int i, int w) {
    const int lo = w * 32;
    if (i < lo) return 0u;
    if (i >= lo + 31) return 0xFFFFFFFFu;
    return (2u << (i - lo)) - 1u;
}

// one element: column rel relative to the draft block (< 0 = the past)
template <typename E>
__device__ __forceinline__ E mask_value(const uint32_t *bits, int rel, int T, E neg) {
    if (rel < 0) return (E)0;
    if (rel >= T) return neg;
    return (bits[rel >> 5] >> (rel & 31)) & 1u ? (E)0 : neg;
}

template <int ES>
__global__ void __launch_bounds__(ASM_THREADS, 4) draft_assemble_kernel(AsmParams p, uint32_t neg) {
    typedef typename MaskBits<ES>::T E;
    constexpr int VEC = 16 / ES;
    __shared__ uint32_t s_anc[ASM_MAX_T][ASM_WORDS];
    __shared__ uint32_t s_row[ASM_ROWS][ASM_WORDS];
    __shared__ int s_par[ASM_MAX_T];
    __shared__ int s_n, s_tree, s_done, s_cl;
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int T = p.T, W = (T + 31) >> 5;
    const int row0 = blockIdx.x * ASM_ROWS;
    const int m_cap = min(T, row0 + ASM_ROWS);    // this tile's rows need the ancestor sets of nodes < m_cap at most
    // the request's header and (speculatively: a stale tree is valid memory) its parents, issued together - one round trip
    if (tid == 0) {
        const int done = p.done ? p.done[b] : 0, ty = p.type ? p.type[b] : SAMD_DRAFT_DYN_SEQ;
        const int tn = p.tree_n ? p.tree_n[b] : 0, dl = p.draft_len[b];
        s_cl = p.cache_len[b];
        // any type but SAMD_DRAFT_STATIC_TREE is a sequence; a non-tree request's tree outputs are stale and never used
        const int tree = p.tree_tok && ty == SAMD_DRAFT_STATIC_TREE;
        int n;
        if (done) n = 1;                                                   // finished: a one-node draft, no path
        else if (tree) n = min(min(tn, p.tree_stride), T);
        else n = min(min(dl, p.draft_stride), min(T, p.D));
        s_n = max(n, 1);
        s_tree = tree;
        s_done = done != 0;
    }
    if (p.tree_tok)
        for (int i = tid; i < min(m_cap, p.tree_stride); i += ASM_THREADS) {
            const int par = p.tree_par[(size_t)b * p.tree_stride + i];
            s_par[i] = (par >= 0 && par < i) ? par : -1;                   // parents precede children
        }
    __syncthreads();
    const int n = s_n, tree = s_tree, done = s_done, cl = s_cl;
    const bool tree_rows = tree && !done;          // rows i < n follow the tree's ancestor sets

    // ---- ancestor sets of the nodes below this tile's last row (a tree tile only) ---------------------------------------
    // A node's set is its parent's set plus itself; unrolled, the chain of its parents.  Every (node, word) pair walks its
    // chain through the parents in shared memory on its own thread: no barrier per tree level.
    if (tree_rows && row0 < n) {
        const int m = min(n, m_cap);
        for (int e = tid; e < m * W; e += ASM_THREADS) {
            const int i = e / W, w = e - i * W;
            uint32_t bits = (i >> 5) == w ? 1u << (i & 31) : 0u;
            for (int j = s_par[i]; j >= 0; j = s_par[j])
                if ((j >> 5) == w) bits |= 1u << (j & 31);
            s_anc[i][w] = bits;
        }
        __syncthreads();
    }

    // ---- the request's small outputs (tile 0) -------------------------------------------------------------------------
    if (blockIdx.x == 0) {
        const size_t o = (size_t)b * T;
        for (int i = tid; i < T; i += ASM_THREADS) {
            int tok = 0, dep = i;
            if (i < n) {
                if (tree) {
                    tok = p.tree_tok[(size_t)b * p.tree_stride + i];
                    if (!done) dep = i == 0 ? 0 : p.tree_dep[(size_t)b * p.tree_stride + i];
                } else {
                    tok = p.draft[(size_t)b * p.draft_stride + i];
                }
            }
            p.tokens[o + i] = tok;
            p.pos[o + i] = (long long)cl + dep;
        }
        int leaves = 1, width = 0;
        if (tree_rows) {
            leaves = min(min(p.tree_shape[2 * b], p.tree_paths), p.P);
            width = min(p.tree_depth, p.D);
        }
        const int PD = p.P * p.D;
        int32_t *ret = p.retrieve + (size_t)b * PD;
        for (int e = tid; e < PD; e += ASM_THREADS) {
            const int r = e / p.D, c = e - r * p.D;
            int v = -1;
            if (tree_rows) {
                if (r < leaves && c < width) v = p.tree_ret[((size_t)b * p.tree_paths + r) * p.tree_depth + c];
            } else if (r == 0 && c < n) {
                v = c;                                   // the sequence's identity path (done: [0, -1, ...])
            }
            ret[e] = v;
        }
        if (tid == 0) {
            p.n_nodes[b] = n;
            // no path for a finished request: the verify walk accepts nothing and maps index 0 -> 0, so no KV row moves
            p.n_paths[b] = done ? 0 : leaves;
        }
    }

    // ---- the mask rows: one warp per row, 16-byte stores --------------------------------------------------------------
    const int i = row0 + warp;
    if (i >= T) return;
    if (lane < W) {
        uint32_t v;
        if (i >= n) v = (i >> 5) == lane ? 1u << (i & 31) : 0u;        // pad row: the past and itself
        else if (tree_rows) v = s_anc[i][lane];
        else v = prefix_word(i, lane);
        s_row[warp][lane] = v;
    }
    __syncwarp();
    const uint32_t *bits = s_row[warp];
    const int kv = p.kv_len;
    E *row = reinterpret_cast<E *>(p.mask) + ((size_t)b * T + i) * (size_t)kv;
    const E NEG = (E)neg;
    // elements before the first 16-byte boundary, the vectors, the tail
    const int head = min(kv, (int)(((16u - ((uint32_t)(uintptr_t)row & 15u)) & 15u) / ES));
    const int n_vec = (kv - head) / VEC;
    const int tail0 = head + n_vec * VEC;
    if (lane < head) row[lane] = mask_value<E>(bits, lane - cl, T, NEG);
    for (int t = tail0 + lane; t < kv; t += 32) row[t] = mask_value<E>(bits, t - cl, T, NEG);
    uint4 *vrow = reinterpret_cast<uint4 *>(row + head);
    const uint32_t fill = ES == 2 ? (neg | (neg << 16)) : neg;
    for (int k = lane; k < n_vec; k += 32) {
        const int rel = head + k * VEC - cl;                  // the vector's first column, relative to the draft block
        uint4 v;
        if (rel + VEC <= 0) {                                  // wholly in the past
            v = make_uint4(0u, 0u, 0u, 0u);
        } else if (rel >= T) {                                 // wholly past the draft block
            v = make_uint4(fill, fill, fill, fill);
        } else if (ES == 2) {
            v.x = (uint32_t)mask_value<E>(bits, rel + 0, T, NEG) | ((uint32_t)mask_value<E>(bits, rel + 1, T, NEG) << 16);
            v.y = (uint32_t)mask_value<E>(bits, rel + 2, T, NEG) | ((uint32_t)mask_value<E>(bits, rel + 3, T, NEG) << 16);
            v.z = (uint32_t)mask_value<E>(bits, rel + 4, T, NEG) | ((uint32_t)mask_value<E>(bits, rel + 5, T, NEG) << 16);
            v.w = (uint32_t)mask_value<E>(bits, rel + 6, T, NEG) | ((uint32_t)mask_value<E>(bits, rel + 7, T, NEG) << 16);
        } else {
            v = make_uint4(mask_value<E>(bits, rel, T, NEG), mask_value<E>(bits, rel + 1, T, NEG),
                           mask_value<E>(bits, rel + 2, T, NEG), mask_value<E>(bits, rel + 3, T, NEG));
        }
        vrow[k] = v;
    }
}

extern "C" int samd_draft_assemble(const samd_assemble_args *a, void *stream) {
    SAMD_REQUIRE(a, "samd_draft_assemble: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->batch <= 65535, "samd_draft_assemble: batch must be in [1, 65535]");
    SAMD_REQUIRE(a->n_nodes > 0 && a->n_nodes <= ASM_MAX_T, "samd_draft_assemble: n_nodes (T) must be in [1, 256]");
    SAMD_REQUIRE(a->n_paths > 0 && a->depth > 0, "samd_draft_assemble: the path table needs n_paths > 0 and depth > 0");
    SAMD_REQUIRE(a->kv_len >= a->n_nodes, "samd_draft_assemble: kv_len must be >= n_nodes (the draft rows are keys too)");
    SAMD_REQUIRE(a->mask_dtype == SAMD_DTYPE_BF16 || a->mask_dtype == SAMD_DTYPE_FP16 || a->mask_dtype == SAMD_DTYPE_FP32,
                 "samd_draft_assemble: mask dtype must be SAMD_DTYPE_BF16 / FP16 / FP32");
    SAMD_REQUIRE(a->draft_dev && a->draft_len_dev && a->draft_stride > 0 && a->cache_len_dev,
                 "samd_draft_assemble: the sequence drafts (draft, draft_len, draft_stride) and cache_len are required");
    SAMD_REQUIRE(a->out_tokens_dev && a->out_position_ids_dev && a->out_n_nodes_dev && a->out_n_paths_dev &&
                 a->out_retrieve_dev && a->out_mask_dev, "samd_draft_assemble: every output is required");
    if (a->tree_tokens_dev) {
        SAMD_REQUIRE(a->type_dev && a->tree_parents_dev && a->tree_depth_dev && a->tree_n_dev && a->tree_retrieve_dev &&
                     a->tree_shape_dev, "samd_draft_assemble: tree drafts need type, parents, depth, n, retrieve and shape");
        SAMD_REQUIRE(a->tree_stride > 0 && a->tree_stride <= a->n_nodes,
                     "samd_draft_assemble: tree_stride must be in [1, n_nodes] (every tree must fit the node rows)");
        SAMD_REQUIRE(a->tree_max_paths > 0 && a->tree_max_paths <= a->n_paths && a->tree_max_depth > 0 &&
                     a->tree_max_depth <= a->depth, "samd_draft_assemble: the tree path table must fit the P x D table");
    }
    AsmParams p;
    p.B = a->batch, p.T = a->n_nodes, p.P = a->n_paths, p.D = a->depth, p.kv_len = a->kv_len;
    p.type = a->type_dev, p.draft = a->draft_dev, p.draft_len = a->draft_len_dev, p.draft_stride = a->draft_stride;
    p.tree_tok = a->tree_tokens_dev, p.tree_par = a->tree_parents_dev, p.tree_dep = a->tree_depth_dev;
    p.tree_n = a->tree_n_dev, p.tree_ret = a->tree_retrieve_dev, p.tree_shape = a->tree_shape_dev;
    p.tree_stride = a->tree_stride, p.tree_paths = a->tree_max_paths, p.tree_depth = a->tree_max_depth;
    p.cache_len = a->cache_len_dev, p.done = a->done_dev;
    p.tokens = a->out_tokens_dev, p.pos = reinterpret_cast<long long *>(a->out_position_ids_dev);
    p.n_nodes = a->out_n_nodes_dev, p.n_paths = a->out_n_paths_dev, p.retrieve = a->out_retrieve_dev, p.mask = a->out_mask_dev;
    const dim3 grid((a->n_nodes + ASM_ROWS - 1) / ASM_ROWS, a->batch);
    cudaStream_t s = (cudaStream_t)stream;
    switch (a->mask_dtype) {
        case SAMD_DTYPE_FP16: draft_assemble_kernel<2><<<grid, ASM_THREADS, 0, s>>>(p, 0xFBFFu); break;
        case SAMD_DTYPE_BF16: draft_assemble_kernel<2><<<grid, ASM_THREADS, 0, s>>>(p, 0xFF7Fu); break;
        default: draft_assemble_kernel<4><<<grid, ASM_THREADS, 0, s>>>(p, 0xFF7FFFFFu); break;
    }
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
