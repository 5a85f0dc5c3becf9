/* pangnn_b200.h — C ABI of the B200-native panGNN message-passing hot path.
 *
 * The reference (fischer-hub/panGNN) is pure Python and has NO plugin / FFI seam (SURVEY.md §8b):
 * its hot path runs through third-party PyTorch-Geometric ops and Python dict loops.  This header
 * is the seam a maintainer binds instead (ctypes stub in INTEGRATION.md); every entry point cites
 * the reference interface it replaces (paths relative to the reference repo).
 *
 * Conventions
 *   - every function returns 0 on success, a negative PANGNN_E* code on failure;
 *     pangnn_last_error() returns a thread-local message.  Nothing throws across the ABI.
 *   - all data pointers are DEVICE pointers owned by the caller and valid for the duration of the
 *     call; scalars are passed by value.  `stream` is a cudaStream_t passed as void*.
 *   - no internal allocation: functions that need scratch take (ws, ws_bytes) and have a
 *     *_workspace_bytes() query.  No global mutable state; re-entrant across streams.
 *   - node ids are int32 (N <= 5e7 < 2^31); row pointers / edge counts are int64.
 *   - calls are asynchronous on `stream`; the caller synchronises.
 */
#ifndef PANGNN_B200_H
#define PANGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PANGNN_ABI_VERSION 4

#define PANGNN_OK 0
#define PANGNN_EINVAL (-1)    /* bad argument (null pointer, unsupported width, ...) */
#define PANGNN_EWORKSPACE (-2) /* workspace too small */
#define PANGNN_ECUDA (-3)     /* CUDA runtime error (message in pangnn_last_error) */

#define PANGNN_ACT_NONE 0
#define PANGNN_ACT_ELU 1

int pangnn_abi_version(void);
const char *pangnn_last_error(void);
/* sha256 of the sources / headers / flags the library was compiled from (pangnn_b200/build.py stamps it in);
 * the Python loader refuses a library that is older than the sources beside it. */
const char *pangnn_source_digest(void);

/* ------------------------------------------------------------------------------------------------
 * Device primitives: LSD radix sort (8-bit digits, stable), exclusive scan, stream compaction.
 * They replace the Python set / dict / list loops of src/helper.py:420-433 (remove_duplicate_edges_tuple),
 * src/preprocessing.py:73-118 (build_edge_index) and the pandas groupby of src/preprocessing.py:413-416.
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_sort_pairs_workspace_bytes(int64_t n);
/* Sorts (key, val) pairs by key bits [0, key_bits).  keys_out/vals_out receive the result;
 * keys_in/vals_in are left untouched.  vals_in may be NULL (then vals = 0..n-1). n < 2^32. */
int pangnn_sort_pairs_u64(const uint64_t *keys_in, const uint32_t *vals_in, uint64_t *keys_out,
                          uint32_t *vals_out, int64_t n, int key_bits, void *ws, size_t ws_bytes,
                          void *stream);

size_t pangnn_scan_workspace_bytes(int64_t n);
/* out[i] = sum_{j<i} in[j]; total (optional, device) = sum of all.  in == out allowed. */
int pangnn_exclusive_scan_u32(const uint32_t *in, uint32_t *out, int64_t n, uint32_t *total,
                              void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * CSR build from a COO edge list (reference: the PyG-style int64 `edge_index` [2,E] that
 * src/dataset.py:282-310,349-384 assembles and torch_geometric.nn.GCNConv consumes at
 * src/gnn.py:129-165).  Rows are destinations when by_dst != 0 (forward aggregation), sources
 * otherwise (the transposed graph used by the backward pass).  Within a row, columns are sorted
 * ascending (canonical order, SURVEY.md F10); duplicates are kept (GCNConv does not coalesce).
 *   rowptr [N+1] int64, col [E] int32, perm [E] uint32 (csr position -> original edge position).
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_csr_build_workspace_bytes(int64_t num_edges);
int pangnn_csr_build(const int64_t *edge_index /* [2,E] row-major: src row then dst row */,
                     int64_t num_edges, int32_t num_nodes, int by_dst, int64_t *rowptr, int32_t *col,
                     uint32_t *perm, void *ws, size_t ws_bytes, void *stream);

/* Edge lists already in canonical (src, dst) order (what this package's preprocessing emits) need no sort for the
 * by-source orientation.  pangnn_edges_sorted: *flags (device) bit 0 = the list is NOT in non-decreasing
 * (src, dst) order, bit 1 = some endpoint lies outside [0, num_nodes) (torch's index ops would raise on such a
 * list; the caller must).  pangnn_csr_from_sorted: by-source CSR of a sorted, in-range list (perm = identity),
 * identical to pangnn_csr_build(by_dst = 0). */
int pangnn_edges_sorted(const int64_t *edge_index, int64_t num_edges, int32_t num_nodes, int32_t *flags,
                        void *stream);
int pangnn_csr_from_sorted(const int64_t *edge_index, int64_t num_edges, int32_t num_nodes, int64_t *rowptr,
                           int32_t *col, uint32_t *perm, void *stream);

/* CSR of the other orientation from an existing one (rows <-> columns): identical to pangnn_csr_build of the
 * same edge list with by_dst flipped (same canonical order, same perm), in ceil(log2 N / 8) radix passes
 * instead of ceil(2 log2 N / 8).  Workspace: pangnn_csr_build_workspace_bytes(num_edges). */
int pangnn_csr_transpose(const int64_t *rowptr, const int32_t *col, const uint32_t *perm, int64_t num_edges,
                         int32_t num_nodes, int64_t *rowptr_t, int32_t *col_t, uint32_t *perm_t, void *ws,
                         size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * gcn_norm (torch_geometric gcn_norm with add_self_loops=False, recomputed inside every GCNConv
 * call at src/gnn.py:129-165): deg[i] = sum_{e: dst_e = i} w_e (sorted-segment sum, fp64
 * accumulate, no atomics), dis = deg^-1/2 (0 where deg == 0), val_e = dis[src]*w_e*dis[dst].
 * `w` is in ORIGINAL edge order (NULL = all ones, the unweighted calls at src/gnn.py:138,165).
 * pangnn_gcn_norm works on the by-destination CSR and emits dis[N] + val[E] in that CSR's order;
 * pangnn_gcn_norm_apply re-emits val for any other ordering of the same edges (the transposed CSR).
 * ---------------------------------------------------------------------------------------------- */
int pangnn_gcn_norm(const int64_t *rowptr, const int32_t *col, const uint32_t *perm, const float *w,
                    int32_t num_nodes, float *dis, float *val, void *stream);
int pangnn_gcn_norm_apply(const int64_t *rowptr, const int32_t *col, const uint32_t *perm,
                          const float *w, const float *dis, int32_t num_nodes, int rows_are_dst,
                          float *val, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Normalised aggregation  Y[i,:] = act( sum_{e in row i} val_e * X[col_e,:] + bias )
 * = GCNConv.propagate + bias (+ the ELU of src/gnn.py:108,130-166) on the by-destination CSR;
 * the same kernel on the transposed CSR is the backward of propagate (SURVEY.md §3.5), and with
 * val == NULL (ones) it is the sorted-segment reduction that returns the edge scorer's per-edge
 * gradients to the nodes.  F (feature width) must be a multiple of 4, <= 512; ldx/ldy are row
 * strides in floats (multiples of 4).  bias may be NULL.  col == NULL (with val == NULL, F in {32,64,128}) means
 * identity columns: entry i of the CSR is row i of X — per-edge rows that already lie in segment order (an edge list
 * in canonical (src, dst) order, reduced by source) are summed without the index stream.
 * ---------------------------------------------------------------------------------------------- */
int pangnn_gcn_aggregate(const int64_t *rowptr, const int32_t *col, const float *val, const float *x,
                         int64_t ldx, int32_t num_rows, int32_t feat, const float *bias, int act,
                         float *y, int64_t ldy, void *stream);

/* ELU backward fused with the bias gradient: g = dy * (y > 0 ? 1 : y + 1), dbias_partial[b,:] =
 * column sums of block b's rows (deterministic two-stage reduce; final sum by the caller or by
 * pangnn_reduce_partials).  Replaces autograd's elu_backward + sum (pangnn.py:207). act as above. */
int pangnn_act_bwd_bias(const float *dy, const float *y, int64_t num_rows, int32_t feat, int act,
                        float *g, float *dbias /* [feat], overwritten */, void *ws, size_t ws_bytes,
                        void *stream);
size_t pangnn_act_bwd_bias_workspace_bytes(int64_t num_rows, int32_t feat);

/* ------------------------------------------------------------------------------------------------
 * Tall-skinny weight-gradient GEMM  C[M,K] = A^T B  (A: [N,M] row stride lda, B: [N,K] row stride
 * ldb, M and K in {64, 128}): dW = dH^T X of every GCN layer and of the hoisted scorer layer
 * (autograd's mm backward behind pangnn.py:207).  Deterministic two-stage reduction over N.
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_gemm_tn_workspace_bytes(int64_t num_rows, int32_t m, int32_t k);
int pangnn_gemm_tn(const float *a, int64_t lda, const float *b, int64_t ldb, int64_t num_rows,
                   int32_t m, int32_t k, float *c, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Node linear transform  Y[M,n] = act(X[M,k] W^T + b)  on the tcgen05 tensor cores with the 3xTF32
 * split (fp32-grade accuracy).  Replaces the `lin` of every torch_geometric GCNConv call
 * (src/gnn.py:129-165), linear_out (src/gnn.py:104,148), the first scorer layer hoisted to the nodes
 * (src/gnn.py:110,177) and, with w_is_kn = 1, the dX = dY W products of their backward
 * (pangnn.py:207).  n, k in {64, 128}.  W is [n, k] row-major (row stride ldw) when w_is_kn = 0 and
 * [k, n] row-major when w_is_kn = 1.  bias may be NULL; act as in pangnn_gcn_aggregate.
 * ---------------------------------------------------------------------------------------------- */
int pangnn_node_linear(const float *x, int64_t ldx, int64_t num_rows, int32_t k, const float *w,
                       int64_t ldw, int w_is_kn, int32_t n, const float *bias, int act, float *y,
                       int64_t ldy, void *stream);
/* Same, fused with the forward halo exchange of the genome-partitioned path (GEMM -> all-gather over
 * NVLink peer memory): every output row r with push_slot{0,1}[r] >= 0 is also stored into row
 * push_slot{0,1}[r] of peer_y{0,1} — the neighbouring rank's extended activation buffer (symmetric
 * memory, same row stride ldy) — from the same epilogue.  Rows outside [lo, hi) are known not to be
 * pushed (the map is not read for them).  Either map may be NULL. */
int pangnn_node_linear_push(const float *x, int64_t ldx, int64_t num_rows, int32_t k, const float *w,
                            int64_t ldw, int w_is_kn, int32_t n, const float *bias, int act, float *y,
                            int64_t ldy, const int32_t *push_slot0, float *peer_y0, int64_t lo0, int64_t hi0,
                            const int32_t *push_slot1, float *peer_y1, int64_t lo1, int64_t hi1, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Candidate normalisation (src/preprocessing.py:370-385 remove_trivial_cases, :430-443
 * softmax_with_temperature, :454-548 normalize_sim_scores) fused with edge-index / weight / label
 * emission (:73-118 build_edge_index, :264-325 map_edge_weights, :122-156 map_labels_to_edge_index).
 *
 * Input: hit table sorted by (query, target) with unique pairs (see pangnn_sort_pairs_u64 and
 * pangnn_hits_dedupe_last), node ids genome-major so that a query's candidates of one genome are
 * contiguous.  Segment = (query, genome_of[target]).  fp64 internally, fp32 out.
 *   pangnn_hits_sort_unique: radix sort by (query, target), duplicate pairs collapse to the LAST
 *            input row (dict(zip) semantics); emits the unique sorted table and its length (device).
 *   pangnn_hits_normalize: segment heads -> scan -> one warp per segment:
 *            keep = 0 for self hits, and (when drop_trivial) for every member of a segment whose
 *            size INCLUDING the self hit is 1;   w = -10 log10(clip(1-p, eps, 1-eps)) + pseudo
 *            with p = softmax(bits/temp) over the non-self members (p = 1 if fewer than 2);
 *            y = (group_of[q] == group_of[t] >= 0)  (group_of may be NULL -> y = 0);
 *            then stream compaction by keep -> (src, dst, w, y) sorted by (src, dst), count (device).
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_hits_sort_unique_workspace_bytes(int64_t num_hits);
int pangnn_hits_sort_unique(const int32_t *q, const int32_t *t, const double *bits, int64_t num_hits,
                            int32_t num_nodes, int32_t *q_out, int32_t *t_out, double *bits_out,
                            uint32_t *count /* device */, void *ws, size_t ws_bytes, void *stream);
size_t pangnn_hits_normalize_workspace_bytes(int64_t num_hits);
int pangnn_hits_normalize(const int32_t *q, const int32_t *t, const double *bits, int64_t num_hits,
                          const int32_t *genome_of, const int32_t *group_of, double temp, double eps,
                          double pseudo, int drop_trivial, int32_t *src, int32_t *dst, float *w,
                          float *y, uint32_t *count /* device */, void *ws, size_t ws_bytes,
                          void *stream);

/* ------------------------------------------------------------------------------------------------
 * Halo exchange of the genome-partitioned multi-GPU path over NVLink PEER memory (new; the reference's
 * only parallelism is implicit DDP, SURVEY §2a / §8e).  `dst` of the first and `src` of the second call
 * are peer device pointers (symmetric-memory mappings); rows are `feat` floats, feat % 4 == 0.
 *   pangnn_rows_gather_copy:  dst[k] = src[idx[k]]      (idx NULL -> k)   forward halo push
 *   pangnn_rows_scatter_add:  dst[idx[k]] += src[k]     (idx unique)      backward halo-gradient pull
 * ---------------------------------------------------------------------------------------------- */
int pangnn_rows_gather_copy(const float *src, int64_t ld_src, const int32_t *idx, int64_t n, int32_t feat, float *dst,
                            int64_t ld_dst, void *stream);
int pangnn_rows_scatter_add(const float *src, int64_t ld_src, const int32_t *idx, int64_t n, int32_t feat, float *dst,
                            int64_t ld_dst, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Data-parallel gradient average over NVLink PEER memory (new; the all-reduce DDP runs behind
 * accelerator.backward, pangnn.py:207).  Every rank of a group of `world` ranks calls push, then reduce, on
 * its stream, the same number of times; both are legal inside a CUDA-graph capture and correct on replay.
 *   grads [count] / numels [count]: host arrays of this rank's gradient tensors (fp32, dense, any size and
 *     alignment; a NULL entry packs zeros and is not written back).  The pointers travel BY VALUE in the
 *     kernel parameters (count <= PANGNN_GRAD_REDUCE_MAX_TENSORS), so no pointer table lives in device memory.
 *   bucket: this rank's symmetric buffer of 2 * half_floats floats (two halves), half_floats >=
 *     pangnn_grad_bucket_floats(numels, count); peer_buckets [world]: every rank's bucket, mapped here.
 *   signal: this rank's symmetric int32 [world] array; peer_signals [world]: every rank's, mapped here.
 *   ctrl: this rank's int32 [4] in ordinary device memory, zeroed once together with `signal` before the
 *     first call: {epoch e, push ticket, reduce ticket, status}.
 *   push:   pack the gradients into half e & 1 of `bucket`; the last CTA then stores e + 1 into
 *           peer_signals[p][rank] of every p (release, system scope).
 *   reduce: wait until signal[0 .. world) >= e + 1 (acquire, %globaltimer budget timeout_ns), then
 *           grad = (b_0 + b_1 + ... + b_{world-1}) * fp32(1 / world), the sum strictly in rank order over
 *           half e & 1 of every peer bucket; the last CTA stores e + 1 into ctrl[0].  On expiry the kernel
 *           stores 1 + (the first rank whose signal is missing) into ctrl[3] and returns without writing.
 * Two halves need one signal per call: a rank that writes half h at call k + 2 has seen every peer's call k + 1
 * signal, which each peer sends only after its call-k reads.  Epoch and parity live in device memory and the
 * signals only grow, so eager calls and replays of different graphs interleave in any order.
 * ---------------------------------------------------------------------------------------------- */
#define PANGNN_GRAD_REDUCE_MAX_TENSORS 32
#define PANGNN_GRAD_REDUCE_MAX_RANKS 8
int64_t pangnn_grad_bucket_floats(const int64_t *numels, int32_t count);
int pangnn_grad_push(float *const *grads, const int64_t *numels, int32_t count, float *bucket, int64_t half_floats,
                     int32_t *const *peer_signals, int32_t world, int32_t rank, int32_t *ctrl, void *stream);
int pangnn_grad_reduce(float *const *grads, const int64_t *numels, int32_t count, const float *const *peer_buckets,
                       int64_t half_floats, const int32_t *signal, int32_t world, int32_t rank, int32_t *ctrl,
                       int64_t timeout_ns, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Whole-graph neighbour band (SURVEY §8 a8; replaces the Python double loop of src/dataset.py:351-366):
 * edges i -> j, j in [i-n, i+n] ∩ [0, N), self loop included, in the reference's loop order.
 * pangnn_neighbour_band_edges is host arithmetic: (2n+1) N - n (n+1) for N > n.  out_src / out_dst are
 * separate so the band can land in the tail of a union edge list (a11, src/dataset.py:373-381).
 * ---------------------------------------------------------------------------------------------- */
int64_t pangnn_neighbour_band_edges(int64_t num_nodes, int32_t n);
int pangnn_neighbour_band(int64_t num_nodes, int32_t n, int64_t *out_src, int64_t *out_dst, void *stream);
/* CSR of the whole-graph union list [sim ; band] (a11) from the CSR of the sim edges alone: every row is
 * merged with its band columns; equals pangnn_csr_build of the concatenated list (perm of a band edge =
 * num_edges + its position in the band), without sorting it.  rowptr_u [N+1], col_u / perm_u [E + band]. */
int pangnn_csr_merge_band(const int64_t *rowptr, const int32_t *col, const uint32_t *perm, int64_t num_edges,
                          int64_t num_nodes, int32_t n, int by_dst, int64_t *rowptr_u, int32_t *col_u,
                          uint32_t *perm_u, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Embedding Linear(1, D) followed by the first GCNConv (src/gnn.py:97,125 then :129 / :135 / :147) as one
 * rank-2 update.  With scalar node features x [N, 1] the embedding E0 = x w_e^T + 1 b_e^T has rank 2 and the
 * convolution is linear in it:  A_hat (E0 W^T) + b = a u^T + c v^T + b,  a = A_hat x, c = A_hat 1 (N-vectors),
 * u = W w_e, v = W b_e (F-vectors).
 *   pangnn_csr_spmv2:        ax[r] = sum_e val_e x[col_e], a1[r] = sum_e val_e  (x NULL = ones; fp64 accumulate)
 *   pangnn_rank1_affine_act: y[r,:] = act(a[r] u + c[r] v + bias)
 *   pangnn_rank1_bwd:        g = dy * act'(y); sums = [sum_r g | sum_r a[r] g | sum_r c[r] g]  ([3, feat];
 *                            per-block partials summed in fixed order, no atomics)
 * ---------------------------------------------------------------------------------------------- */
int pangnn_csr_spmv2(const int64_t *rowptr, const int32_t *col, const float *val, const float *x, int32_t num_rows,
                     float *ax, float *a1, void *stream);
int pangnn_rank1_affine_act(const float *a, const float *c, const float *u, const float *v, const float *bias,
                            int64_t num_rows, int32_t feat, int act, float *y, int64_t ldy, void *stream);
size_t pangnn_rank1_bwd_workspace_bytes(int64_t num_rows, int32_t feat);
int pangnn_rank1_bwd(const float *dy, const float *y, const float *a, const float *c, int64_t num_rows, int32_t feat,
                     int act, float *sums, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Batch collation on the device (SURVEY §8 a12; replaces torch_geometric Batch.from_data_list behind
 * DataLoader, pangnn.py:121,152-153; semantics SURVEY A.3).  The graphs of a split are packed back to back
 * per attribute (`src`, with `seg_ptr[g] .. seg_ptr[g+1]` the items of graph g); a batch is `graph_ids`
 * [batch_size] (device).  Per attribute: items of the batch's graphs are concatenated into `dst` in batch
 * order.  kind INDEX (int64, 2 rows = an `*index*` attribute [2, e]): every value is shifted by the
 * cumulative node count of the preceding graphs of the batch; kind FILL_SLOT writes the graph slot of every
 * item (PyG's `batch` vector; its seg_ptr is the node range table).  `node_attr` names the attribute whose
 * segments are the node ranges (x, or the FILL_SLOT attribute).  `offsets` [num_attrs, batch_size + 1] int64
 * (device, output) receives the exclusive scan of the segment sizes per attribute — row `node_attr` is
 * PyG's `ptr`.  Output sizes are host arithmetic over the caller's copy of the seg_ptr tables.
 * Two launches per batch, independent of the number of attributes.
 * ---------------------------------------------------------------------------------------------- */
#define PANGNN_COLLATE_MAX_ATTRS 12
#define PANGNN_COLLATE_COPY 0
#define PANGNN_COLLATE_INDEX 1
#define PANGNN_COLLATE_FILL_SLOT 2
typedef struct pangnn_collate_attr {
    const void *src;          /* packed attribute (device); NULL for FILL_SLOT */
    const int64_t *seg_ptr;   /* [num_graphs + 1] item offsets per graph (device) */
    void *dst;                /* output (device) */
    int64_t src_row_stride;   /* elements between the rows of a 2-row attribute in src (0 if rows == 1) */
    int64_t dst_row_stride;   /* same in dst = total items of this attribute in the batch */
    int32_t rows;             /* 1 or 2 */
    int32_t elem_bytes;       /* 4 or 8 */
    int32_t kind;             /* PANGNN_COLLATE_* */
    int32_t width;            /* elements per item (x [n, 1] -> 1) */
} pangnn_collate_attr;
int pangnn_collate(const pangnn_collate_attr *attrs /* host */, int32_t num_attrs, int32_t node_attr,
                   const int32_t *graph_ids, int32_t batch_size, int64_t *offsets, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Max-candidate baselines (SURVEY §8f rank 1): calculate_baseline_labels (src/helper.py:437-485) and
 * calculate_logit_baseline_labels / find_max_logit (src/helper.py:494-576) as one segmented arg-max.
 * (q, t) sorted by (query, target) as produced by pangnn_hits_sort_unique / pangnn_hits_normalize;
 * segment = (query, genome_of[target]); label[i] = 1 iff no entry of the segment has a strictly larger
 * score.  score is fp64 (raw bit scores) when score_is_f64 != 0, else fp32 (Q-scores, logits).
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_segment_max_labels_workspace_bytes(int64_t n);
int pangnn_segment_max_labels(const int32_t *q, const int32_t *t, const void *score, int score_is_f64, int64_t n,
                              const int32_t *genome_of, int32_t *label, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused edge scorer (src/gnn.py:110-116,171-177: gather h[src], h[dst] (+ edge_attr[:E]), concat,
 * Linear-ReLU-Linear-ReLU-Linear) with the first layer hoisted to the nodes:
 *     pq[n, 0:D] = h[n] @ W1[:, 0:D]^T,   pq[n, D:2D] = h[n] @ W1[:, D:2D]^T      (node GEMM, caller)
 *     a1 = pq[src,0:D] + pq[dst,D:2D] (+ w1c*skip_e) + b1 ; z = w3 . relu(W2 relu(a1) + b2) + b3
 * D must be 64 (the reference default --node_dim; other widths take the unfused path upstream).
 * fwd writes logits[E]; with y != NULL it also accumulates the BCE-with-logits(pos_weight) loss SUM
 * (pangnn.py:98,203) into loss_sum (device double, caller zeroes) and the thresholded prediction is
 * left to the caller.
 * bwd recomputes the forward per tile and emits
 *     da1[E,D] (per-edge gradient wrt a1, to be segment-reduced to the nodes),
 *     grads[] = { dW2[D*D], db2[D], dw3[D], db3[1], db1[D], dw1c[D] }  (overwritten).
 * dz comes from dlogits[E] when given, else from the fused BCE:  dz = scale*((1-y)s - pw*y*(1-s)).
 * ---------------------------------------------------------------------------------------------- */
#define PANGNN_SCORER_D 64
#define PANGNN_SCORER_NGRADS (64 * 64 + 64 + 64 + 1 + 64 + 64)
size_t pangnn_edge_score_workspace_bytes(int64_t num_edges);
int pangnn_edge_score_fwd(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                          const float *w1c, const float *b1, const float *w2, const float *b2,
                          const float *w3, const float *b3, int64_t num_edges, const float *y,
                          float pos_weight, float *logits, double *loss_sum, void *ws,
                          size_t ws_bytes, void *stream);
/* logits / loss_sum are optional outputs of the backward pass too (fused training step: one kernel
 * yields logits, loss and every gradient). */
/* Inference form with the prediction head fused in (pangnn.py:220-221,262-263; src/predict.py:54-55):
 * prob = sigmoid(logit), pred = prob >= threshold.  logits / prob / pred may each be NULL. */
int pangnn_edge_score_predict(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                              const float *w1c, const float *b1, const float *w2, const float *b2,
                              const float *w3, const float *b3, int64_t num_edges, float threshold,
                              float *logits, float *prob, int32_t *pred, void *stream);
int pangnn_edge_score_bwd(const float *pq, const int32_t *src, const int32_t *dst, const float *skip,
                          const float *w1c, const float *b1, const float *w2, const float *b2,
                          const float *w3, const float *b3, int64_t num_edges, const float *dlogits,
                          const float *y, float pos_weight, float scale, float *da1, float *grads,
                          float *logits, double *loss_sum, void *ws, size_t ws_bytes, void *stream);

/* Cosine decoder of src/gnn.py:179,206-207 (F.cosine_similarity, eps 1e-8) and the row-wise dot
 * of src/gnn.py:77-79 (mode 0 = cosine, 1 = dot), forward only. */
int pangnn_edge_pair_score(const float *h, int64_t ldh, int32_t feat, const int32_t *src,
                           const int32_t *dst, int64_t num_edges, int mode, float *out, void *stream);

/* Backward of the two decoders above (autograd of src/gnn.py:202-207 at pangnn.py:207): dh [N, feat] (dense,
 * row stride feat) = gradient w.r.t. the node embeddings given dz [E] = gradient w.r.t. the scores and
 * out [E] = the forward scores.  Both CSR orientations of the scored-edge graph (pangnn_csr_build /
 * pangnn_csr_transpose) are walked: the gradient is two weighted aggregations plus a diagonal term, so no per-edge
 * [E, feat] rows are materialised (the reference's autograd gathers and scatters four of them). */
size_t pangnn_edge_pair_score_bwd_workspace_bytes(int64_t num_edges, int32_t num_nodes, int32_t feat);
int pangnn_edge_pair_score_bwd(const float *h, int64_t ldh, int32_t feat, int32_t num_nodes, int64_t num_edges,
                               const int64_t *rowptr_src, const int32_t *col_src, const uint32_t *perm_src,
                               const int64_t *rowptr_dst, const int32_t *col_dst, const uint32_t *perm_dst,
                               const float *dz, const float *out, int mode, float *dh, void *ws, size_t ws_bytes,
                               void *stream);

/* ------------------------------------------------------------------------------------------------
 * MMseqs2 hit table parser (SURVEY §8f rank 2; replaces pandas read_csv + per-row id lookups of
 * src/preprocessing.py:388-426): the file's bytes are parsed on the device.
 *   pangnn_tsv_line_index: *num_newlines (device) = '\n' count; with line_start != NULL also
 *                          line_start[0] = 0, line_start[k] = offset after the k-th newline (num_newlines + 1
 *                          entries).  Call once with NULL to size the arrays, once more to fill them.
 *   pangnn_tsv_parse_hits: per line (num_lines = num_newlines, + 1 if the text does not end with a newline):
 *                          q / t = node id of column 0 / 1 looked up by FNV-1a-64 hash in the sorted table of
 *                          known gene ids (-1 unknown, -2 blank or '#' line), bits = column score_col as double.
 * ---------------------------------------------------------------------------------------------- */
size_t pangnn_parse_hits_tsv_workspace_bytes(int64_t num_bytes);
int pangnn_tsv_line_index(const uint8_t *text, int64_t num_bytes, int64_t *line_start, int64_t max_lines,
                          uint32_t *num_newlines, void *ws, size_t ws_bytes, void *stream);
int pangnn_tsv_parse_hits(const uint8_t *text, int64_t num_bytes, const int64_t *line_start, int64_t num_lines,
                          int64_t num_newlines, int32_t score_col, const uint64_t *id_hash_sorted,
                          const int32_t *id_pos, int32_t num_ids, int32_t *q, int32_t *t, double *bits,
                          void *stream);

/* ------------------------------------------------------------------------------------------------
 * Output side (SURVEY §8f rank 4): ortholog groups = connected components of the edges predicted positive
 * (intended behaviour of write_groups_file, src/postprocessing.py:5-36, which as written never merges two sets).
 * labels[i] = smallest gene id of i's component.  pangnn_components_init sets labels[i] = i; every
 * pangnn_components_round hooks the selected edges (select NULL = all; otherwise select[e] != 0) and flattens
 * the trees, writing *changed (device) = 1 if any hook happened: repeat until it reads 0.
 * ---------------------------------------------------------------------------------------------- */
int pangnn_components_init(int32_t *labels, int32_t num_nodes, void *stream);
int pangnn_components_round(const int32_t *src, const int32_t *dst, const int32_t *select, int64_t num_edges,
                            int32_t *labels, int32_t num_nodes, int32_t *changed, void *stream);

/* ------------------------------------------------------------------------------------------------
 * GFF3 annotation and RIBAP group table on the device (src/preprocessing.py:329-367 load_gff, :159-193
 * load_ribap_groups; both pandas read_csv(sep = tab, comment = '#') in the reference).  Line index as for the hit
 * table (pangnn_tsv_line_index).
 * pangnn_gff_parse_lines: per line flags (1 record | 2 complete: 9 fields, none missing | 4 attribute mentions
 * start_gene | 8 id matches [A-Z]+_[0-9]+ | 16 "ID=" occurs inside the id: resolve on the host), byte range of the
 * gene id (attribute up to ';' without the leading "ID=") and its FNV-1a 64 hash.  The caller rotates the records to
 * the start gene and compacts (a scan over the flags).
 * pangnn_tsv_lookup_columns: node id of the gene named in every kept column of every line (col_slot[c] = output
 * slot of column c, -1 = ignored): out[line * num_slots + slot] = node id | -1 unknown id | -2 missing cell. */
int pangnn_gff_parse_lines(const uint8_t *text, int64_t num_bytes, const int64_t *line_start, int64_t num_lines,
                           int64_t num_newlines, const uint8_t *start_gene, int32_t start_gene_len, int32_t *flags,
                           int64_t *id_off, int32_t *id_len, uint64_t *id_hash, void *stream);
int pangnn_tsv_lookup_columns(const uint8_t *text, int64_t num_bytes, const int64_t *line_start, int64_t num_lines,
                              int64_t num_newlines, const int32_t *col_slot, int32_t num_cols, int32_t num_slots,
                              const uint64_t *id_hash_sorted, const int32_t *id_pos, int32_t num_ids, int32_t *out,
                              int32_t *line_flag, void *stream);

/* ------------------------------------------------------------------------------------------------
 * --simulate_dataset on the device (src/simulate.py:103-199): the hit table (query, target, bit score) of the
 * queries of genomes [q_lo, q_hi) of an n x G pan-genome, generated by counter-based Philox streams keyed by
 * (seed, genome, gene, draw) — every rank of a genome-partitioned run generates its own slab and agrees with its
 * neighbours on the hits across the seam.  Adjacent genomes only (the default trivial-case filter drops the rest).
 * Step 1: pangnn_simulate_neg_counts -> k[i], the number of negative candidates of source gene i of genomes
 * [g_first, g_first + num_genomes) (clip(NegBin(0.2, 0.2/(m+0.2)), 1, n), src/simulate.py:131-132).  The caller
 * scans k into the row offsets of the forward (query = source) and reverse (query = negative target) blocks.
 * Step 2: pangnn_simulate_edges writes rows [positives | forward negatives | reverse negatives]; a negative that
 * lands on the ortholog position follows the positive, so pangnn_hits_sort_unique (last row wins) reproduces the
 * reference's dict overwrite.  new_of_old: synteny permutation (src/simulate.py:202-230) as new GLOBAL node id of
 * every old node of genomes [new_first_genome, ...). */
int pangnn_simulate_neg_counts(uint64_t seed, int32_t n, int64_t m, int32_t g_first, int32_t num_genomes,
                               uint32_t *k, void *stream);
int pangnn_simulate_edges(uint64_t seed, int32_t n, int32_t G, int32_t q_lo, int32_t q_hi, double neg_mean,
                          double pos_mean, double dispersion, int32_t g_first, int32_t num_src_genomes,
                          const uint32_t *kcnt, const int64_t *fwd_off, const int64_t *rev_off, int64_t num_pos_rows,
                          int64_t num_fwd_rows, const int32_t *new_of_old, int32_t new_first_genome,
                          int32_t *q, int32_t *t, double *bits, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Exact ranking metrics: ROC AUC, average precision and the Youden threshold (the reference computes them with
 * torchmetrics BinaryAUROC / BinaryAveragePrecision every epoch, pangnn.py:27-30,220-222,262-268,279-326, and with
 * sklearn roc_auc_score / average_precision_score / roc_curve at test time, src/plot.py:103-107,131).
 * A "run" is one distinct score with its positive and negative counts; runs are int64 rows (key, pos, neg) in
 * DECREASING score order, key = the score's 32-bit order key (-0.0 and +0.0 share one).
 *   pangnn_metric_runs:   runs of (scores [n] fp32, labels [n] of label_kind) — key pass, pangnn_sort_pairs_u64 on
 *                         32 key bits, compaction — or, with runs_in != NULL, of n input runs in any order (equal
 *                         keys are merged, counts summed; scores / labels ignored).  runs_out has room for n rows.
 *                         info [6] (device, written): runs, P, N, 0, 0, flags (PANGNN_METRIC_*; the caller raises).
 *                         hist (device, optional) [65536]: number of runs per top 16 key bits.  n < 2^32.
 *   pangnn_metric_reduce: over runs with params [5] (device) = (runs, P, N, TP_0, FP_0): P, N the global class
 *                         counts, (TP_0, FP_0) the counts ranked ahead of these runs (0 on one device; info
 *                         serves as params).  max_runs sizes the launch.  out [8] (device):
 *                         [0..1] sum_k neg_k (TP_{k-1} + TP_k) as unsigned 128-bit (lo, hi)  -> AUROC = / (2 P N)
 *                         [2..3] sum_k pos_k floor(TP_k 2^s / (TP_k + FP_k)), 128-bit, s = out[7] = 127 - bitlen(P)
 *                                -> AP = / (P 2^s)
 *                         [4] max_k TP_k/P - FP_k/N (fp64 bits; -inf if P or N is 0), [5] key of the first run that
 *                         reaches it (all ones if none), [6] runs.
 * Integer accumulation throughout: results do not depend on input order, tiling or a split of the runs.
 * ---------------------------------------------------------------------------------------------- */
#define PANGNN_LABEL_F32 0
#define PANGNN_LABEL_I32 1
#define PANGNN_LABEL_I64 2
#define PANGNN_LABEL_U8 3
#define PANGNN_METRIC_NAN 1        /* a score is NaN */
#define PANGNN_METRIC_BAD_LABEL 2  /* a label is not 0 or 1 */
size_t pangnn_metric_runs_workspace_bytes(int64_t n);
int pangnn_metric_runs(const float *scores, const void *labels, int label_kind, const int64_t *runs_in, int64_t n,
                       int64_t *runs_out, int64_t *info, int64_t *hist, void *ws, size_t ws_bytes, void *stream);
size_t pangnn_metric_reduce_workspace_bytes(int64_t max_runs);
int pangnn_metric_reduce(const int64_t *runs, int64_t max_runs, const int64_t *params, int64_t *out, void *ws,
                         size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * ROC and precision-recall curve points over runs (replaces sklearn roc_curve / precision_recall_curve at
 * src/plot.py:103-107,131 of the reference, and the data behind its TensorBoard PR curve).
 *   params [5] (device): as pangnn_metric_reduce.  bound [3] (device): (pos, neg) of the run that follows the last
 *   of these runs in the whole curve, and PANGNN_CURVE_FIRST (these runs start the curve) | PANGNN_CURVE_FOLLOWED
 *   (a run follows them); (0, 0, PANGNN_CURVE_FIRST) on one device.
 *   mode: PANGNN_CURVE_ALL keeps every run; otherwise run k is kept if it is the first or the last of the curve, or
 *   PANGNN_CURVE_ROC: (pos_{k+1}, neg_{k+1}) != (pos_k, neg_k)   (sklearn roc_curve drop_intermediate)
 *   PANGNN_CURVE_PR:  pos_k != 0 or pos_{k+1} != 0               (sklearn precision_recall_curve drop_intermediate)
 *   Kept runs in order: thresholds [c] fp32 (the run's score, +0.0 for the zeros), tp [c] = TP_0 + TP_k,
 *   fp [c] = FP_0 + FP_k (int64); each output has room for max_runs points.  count [3] (device, written): kept
 *   points, positives and negatives of the runs.  Deterministic, no atomics.
 * ---------------------------------------------------------------------------------------------- */
#define PANGNN_CURVE_ALL 0
#define PANGNN_CURVE_ROC 1
#define PANGNN_CURVE_PR 2
#define PANGNN_CURVE_FIRST 1     /* bound[2]: these runs start the curve */
#define PANGNN_CURVE_FOLLOWED 2  /* bound[2]: a run follows the last of them */
size_t pangnn_metric_curve_workspace_bytes(int64_t max_runs);
int pangnn_metric_curve(const int64_t *runs, int64_t max_runs, const int64_t *params, const int64_t *bound, int mode,
                        float *thresholds, int64_t *tp, int64_t *fp, int64_t *count, void *ws, size_t ws_bytes,
                        void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PANGNN_B200_H */
