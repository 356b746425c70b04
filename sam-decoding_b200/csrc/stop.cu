// Stop sequences: samd_stop_match (include/samd_b200.h).
//
// Request b's output so far is hist[0 .. hist_len); this step would emit tokens[0 .. count).  A stop sequence s of
// length L ends at step position i when the output tokens at positions hist_len + i - L + 1 .. hist_len + i equal s
// (no output position before 0).  The step's output then ends at the earliest such i; among the sequences ending there,
// the lowest index wins.
//
// One CTA per request.  It stages the last SAMD_STOP_MAX_LEN - 1 history tokens followed by the candidates in shared
// memory, and the request's table beside them; thread q takes the (end position, sequence) pairs q, q + STOP_THREADS, ...
// of position * SAMD_STOP_MAX_SEQS + index, compares at most SAMD_STOP_MAX_LEN ids each, and a block-wide minimum of the
// matching keys gives the earliest end with the lowest index.  The minimum does not depend on which thread found which
// key, so the result depends only on the inputs.
#include "samd_common.cuh"
#include "../../include/samd_b200.h"

#include <limits.h>

#define STOP_THREADS 256
#define STOP_MAX_WIDTH 256
#define STOP_TAIL (SAMD_STOP_MAX_LEN - 1)

namespace {

__global__ void __launch_bounds__(STOP_THREADS) stop_match_kernel(samd_stop_args A) {
    __shared__ int s_seq[STOP_TAIL + STOP_MAX_WIDTH];              // history tail, then the candidates
    __shared__ int s_stop[SAMD_STOP_MAX_SEQS * SAMD_STOP_MAX_LEN];
    __shared__ int s_len[SAMD_STOP_MAX_SEQS];
    __shared__ int s_warp[STOP_THREADS / 32];

    const int b = blockIdx.x, tid = threadIdx.x;
    const int count = A.count_dev[b];                              // read by every thread before any write below
    const bool live = !(A.done_dev && A.done_dev[b]) && count > 0;
    const int n = live ? min(count, A.width) : 0;
    const int hl = min(max(A.hist_len_dev[b], 0), A.hist_stride);
    const int h = min(hl, STOP_TAIL);                              // history tokens staged: output positions hl - h ..

    if (n > 0) {
        const int32_t *hist = A.hist_dev + (size_t)b * A.hist_stride + (hl - h);
        const int32_t *tok = A.tokens_dev + (size_t)b * A.width;
        for (int k = tid; k < h + n; k += STOP_THREADS) s_seq[k] = k < h ? hist[k] : tok[k - h];
        const int32_t *st = A.stop_tokens_dev + (size_t)b * SAMD_STOP_MAX_SEQS * SAMD_STOP_MAX_LEN;
        for (int k = tid; k < SAMD_STOP_MAX_SEQS * SAMD_STOP_MAX_LEN; k += STOP_THREADS) s_stop[k] = st[k];
        if (tid < SAMD_STOP_MAX_SEQS) s_len[tid] = A.stop_len_dev[(size_t)b * SAMD_STOP_MAX_SEQS + tid];
    }
    __syncthreads();                                               // (count is read by all before out_count is written)

    int best = INT_MAX;
    for (int q = tid; q < n * SAMD_STOP_MAX_SEQS; q += STOP_THREADS) {
        const int i = q / SAMD_STOP_MAX_SEQS, j = q - i * SAMD_STOP_MAX_SEQS;
        const int L = s_len[j];
        const int first = h + i - L + 1;                           // staged index of the sequence's first token
        if (L <= 0 || L > SAMD_STOP_MAX_LEN || first < 0) continue;
        const int *want = s_stop + j * SAMD_STOP_MAX_LEN;
        bool hit = true;
        for (int k = 0; k < L && hit; ++k) hit = s_seq[first + k] == want[k];
        if (hit) best = min(best, q);                              // q = i * SAMD_STOP_MAX_SEQS + j
    }
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(SAMD_FULL, best, o));
    if ((tid & 31) == 0) s_warp[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < STOP_THREADS / 32; ++w) best = min(best, s_warp[w]);
        A.out_count_dev[b] = best == INT_MAX ? count : best / SAMD_STOP_MAX_SEQS + 1;
        A.out_hit_dev[b] = best == INT_MAX ? -1 : best % SAMD_STOP_MAX_SEQS;
    }
}

}  // namespace

extern "C" int samd_stop_match(const samd_stop_args *a, void *stream) {
    SAMD_REQUIRE(a && a->tokens_dev && a->count_dev && a->hist_dev && a->hist_len_dev && a->stop_tokens_dev &&
                 a->stop_len_dev && a->out_count_dev && a->out_hit_dev, "samd_stop_match: bad arguments");
    SAMD_REQUIRE(a->batch > 0 && a->width > 0 && a->width <= STOP_MAX_WIDTH && a->hist_stride > 0,
                 "samd_stop_match: bad shape (width must be in [1, 256])");
    stop_match_kernel<<<a->batch, STOP_THREADS, 0, (cudaStream_t)stream>>>(*a);
    samd_count_launch();
    SAMD_CUDA(cudaGetLastError());
    return 0;
}
