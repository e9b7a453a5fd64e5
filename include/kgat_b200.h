/*
 * kgat_b200.h  --  C ABI of libkgat_b200.so: the sm_100a CUDA kernels behind the KGAT hot path.
 *
 * The reference (Konippi/problem-recommender-system-using-kgat-in-codeforces) is pure Python on top
 * of PyTorch ATen; it has no FFI of its own.  The drop-in boundary is therefore the Python class
 * surface `src.model.KGAT.model.{KGAT, KGATArgs, KGATMode}` (reference src/model/KGAT/model.py:13-431)
 * and this header is what that surface binds underneath: one entry point per ATen call chain it
 * replaces.  Every entry point cites the reference lines whose arithmetic it implements.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked "host";
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no allocation and no global state inside: the caller owns every buffer, incl. workspaces
 *     (sizes from the matching *_workspace_bytes function);
 *   - return 0 on success, a negative KGAT_ERR_* code otherwise (kgat_error_string explains);
 *   - fp32 values, int32 indices inside the graph containers, int64 ids at the model boundary
 *     (`ids64` arguments), row-major dense matrices with an explicit leading dimension where useful.
 *   - all kernels are asynchronous on `stream` except the functions documented as synchronous.
 */
#ifndef KGAT_B200_H_
#define KGAT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGAT_OK 0
#define KGAT_ERR_INVALID_ARGUMENT (-1)
#define KGAT_ERR_CUDA (-2)
#define KGAT_ERR_UNSUPPORTED (-3)
#define KGAT_ERR_WORKSPACE (-4)

#define KGAT_ABI_VERSION 14
#define KGAT_MAX_LAYERS 8   /* embedding table + up to 7 propagation layers */
#define KGAT_MAX_TENSORS 24 /* tensors per multi-tensor Adam launch */
#define KGAT_MAX_PEERS 31   /* other ranks of a row-sharded propagation */
#define KGAT_PEER_HANDLE_BYTES 64

/* ------------------------------------------------------------------------------------------- */
/* misc                                                                                        */
/* ------------------------------------------------------------------------------------------- */
int kgat_abi_version(void);
const char* kgat_error_string(int code);
/* last CUDA error string seen by this library on the calling thread ("" if none) */
const char* kgat_last_cuda_error(void);
/* device properties the host side sizes grids with (synchronous, host out-pointers) */
int kgat_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes);

/* ------------------------------------------------------------------------------------------- */
/* graph containers: replaces torch.sparse COO coalescing (reference model.py:359-364, the      */
/* implicit coalesce inside torch.sparse.softmax) and scipy's coo->csr (preprocess.py:629)      */
/* ------------------------------------------------------------------------------------------- */

/* Group n 64-bit keys (arbitrary order, duplicates allowed).  Stable: entries with equal keys keep
 * their input order inside the group.  Outputs:
 *   order[n]        sorted position -> input entry index
 *   group_of[n]     input entry index -> group id (dense rank of its key, ascending key order)
 *   group_ptr[g+1]  group id -> first sorted position (group_ptr[n_groups] = n)
 *   unique_keys[g]  ascending unique keys
 *   *n_groups_host  number of groups (host pointer)
 * SYNCHRONOUS (returns after the stream has drained; n_groups is needed on the host). */
int64_t kgat_group_by_key_workspace_bytes(int64_t n);
int kgat_group_by_key(const uint64_t* keys, int64_t n, int key_bits, void* workspace, int64_t workspace_bytes,
                      int32_t* order, int32_t* group_of, int32_t* group_ptr, uint64_t* unique_keys,
                      int64_t* n_groups_host, void* stream);

/* Decode ascending unique keys  key = major * n_minor + minor  into a compressed pointer array over
 * `n_major` majors and the minor index of every key (CSR: major=row, minor=col; CSC: swapped). */
int kgat_decode_sorted_keys(const uint64_t* unique_keys, int64_t n_keys, int64_t n_major, int64_t n_minor,
                            int32_t* major_ptr /* n_major+1 */, int32_t* minor_idx /* n_keys */, void* stream);

/* out[g] = sum over sorted positions p in [group_ptr[g], group_ptr[g+1]) of in[order[p]], summed in
 * that order (deterministic duplicate merge: what COO coalescing does, model.py:364). */
int kgat_segment_sum_f32(const float* in, const int32_t* order, const int32_t* group_ptr, int64_t n_groups, float* out,
                         void* stream);

/* out[i] = in[index[i]]  (permute CSR values into CSC order after each attention refresh) */
int kgat_gather_f32(const float* in, const int32_t* index, int64_t n, float* out, void* stream);
/* out[i] = (int32) in[i] with range check against [0, bound): returns KGAT_ERR_INVALID_ARGUMENT
 * through *bad_count_dev (device int32, incremented per offending element) */
int kgat_ids64_to_i32(const int64_t* in, int64_t n, int64_t bound, int32_t* out, int32_t* bad_count_dev, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K1: attentive SpMM  Y = A * X (+ Z)    reference aggregator.py:54 and its autograd transpose  */
/* ------------------------------------------------------------------------------------------- */
/* A in CSR (row_ptr unused: the task list carries the ranges); X: n_cols x d (leading dim ldx; tables
 * under 4 GiB are addressed with 32-bit byte offsets),
 * Y: n_rows x d (ldy); optional addend Z (ldz) or NULL.  d must be a multiple of 4, <= 256.
 * tasks: n_tasks x {row, begin, end, partial_slot}; a row longer than the plan's chunk is split into
 * several tasks with partial_slot >= 0 whose sums go to `partials` (n_partials x d floats) and are
 * reduced in chunk order for heavy_rows[h] = {row, first_partial_slot, n_chunks, arrival counter}
 * by the warp that finishes the row's last chunk (deterministic, no float atomics; the counter column is
 * scratch owned by the kernel: zero on entry, zero on exit).  The plan is host logic (graph.py: spmm_plan). */
int kgat_spmm_csr(const int32_t* tasks, int64_t n_tasks, int32_t* heavy_rows, int64_t n_heavy,
                  const int32_t* col_idx, const float* vals, const float* X, int64_t n_cols, int64_t ldx, float* Y,
                  int64_t ldy, const float* Z, int64_t ldz, int32_t d, float* partials, void* stream);

/* The same product restricted to the rows / edges a TRAIN_CF step actually needs (frontier section below):
 *   row_mask  (bitmap over output rows, NULL = all): tasks of other rows are skipped, their Y rows left untouched;
 *   edge_mask (bitmap over columns,     NULL = all): edges whose column is outside are dropped (their X rows hold no
 *             valid data) and the addend Z[row] is added only for rows inside it.
 * Bit i of a bitmap is bit (i & 31) of word i >> 5. */
int kgat_spmm_csr_masked(const int32_t* tasks, int64_t n_tasks, int32_t* heavy_rows, int64_t n_heavy,
                         const int32_t* col_idx, const float* vals, const float* X, int64_t n_cols, int64_t ldx, float* Y,
                         int64_t ldy, const float* Z, int64_t ldz, int32_t d, float* partials, const uint32_t* row_mask,
                         const uint32_t* edge_mask, void* stream);

/* Persistent variant over a needed-row LIST (one warp strides over work items; no CTA is launched for a dead row):
 * work = the plan's first n_heavy_tasks tasks (the chunks of the heavy rows; filtered by row_mask, required then) followed
 * by rows[0 .. *n_rows_dev) where a light row owns the single task n_heavy_tasks + light_rank[row] (light_rank[row] < 0
 * marks a heavy row); rows == NULL runs every task (dense output, e.g. the embedding gradient) and only masks edges.
 * edge_mask as above (staged in shared memory when n_mask_bits / 8 <= 32 KB).  d in {16, 32, 64, 128}. */
int kgat_spmm_csr_rows(const int32_t* tasks, int64_t n_tasks, int64_t n_heavy_tasks, const int32_t* light_rank,
                       int32_t* heavy_rows, int64_t n_heavy, const int32_t* col_idx, const float* vals, const float* X,
                       int64_t n_cols, int64_t ldx, float* Y, int64_t ldy, const float* Z, int64_t ldz, int32_t d,
                       float* partials, const int32_t* rows, const int32_t* n_rows_dev, const uint32_t* row_mask,
                       const uint32_t* edge_mask, int64_t n_mask_bits, void* stream);

/* Transposed product as a scatter over a needed-row list:  Y[c] += A[r, c] * G[r] for the *n_rows_dev listed rows r and
 * their edges, and Y[r] += Z[r] (Z nullable) -- 128-bit vector reductions, so Y's destination rows must be zero on entry
 * (kgat_frontier_zero_rows) and the fp32 summation order is not fixed.  tasks / n_heavy_tasks / light_rank / row_mask: the
 * plan of A (not of its transpose) and the list's bitmap, as in kgat_spmm_csr_rows.  d in {16, 32, 64, 128}. */
int kgat_spmm_scatter_rows(const int32_t* tasks, int64_t n_heavy_tasks, const int32_t* light_rank, const int32_t* rows,
                           const int32_t* n_rows_dev, int64_t max_rows, const uint32_t* row_mask, const int32_t* col_idx,
                           const float* vals, const float* G, int64_t ldg, const float* Z, int64_t ldz, float* Y, int64_t ldy,
                           int32_t d, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Needed-row frontier of a TRAIN_CF step: exact pruning of model.py:188 (the full propagation   */
/* is re-run per mini-batch although model.py:189-191 gathers only the <= 3B batch rows)         */
/* ------------------------------------------------------------------------------------------- */
/* F_L = {batch ids}, F_{l-1} = F_l U cols(A[F_l, :]): layer l is computed for the rows of F_l only; every row outside
 * has an exactly-zero gradient and is never read, so loss and gradients equal the reference's.  A level is a bitmap
 * over the nodes plus the ascending list of its rows with a device-side count (everything stream-ordered). */
/* Membership is collected in `flags`, one BYTE per node (32 * ceil(n_nodes / 32) bytes, 16-byte aligned, all zero between
 * builds) with plain idempotent stores, then folded into the level's bitmap by kgat_frontier_list, which clears the flags. */
/* flags[ids64[i]] = 1; ids outside [0, n_nodes) are skipped and counted in *bad_count_dev (nullable) */
int kgat_frontier_mark_ids(const int64_t* ids64, int64_t n_ids, int64_t n_nodes, uint8_t* flags, int32_t* bad_count_dev,
                           void* stream);
/* flags[r] = flags[c] = 1 for the *count_dev rows r listed in `rows` (their bitmap: level_bitmap) and every column c of
 * A[r, :].  Work items are the SpMM plan's tasks (kgat_spmm_csr_rows: the first n_heavy_tasks chunk tasks filtered by
 * level_bitmap, then the listed light rows through light_rank), so hub rows are spread over many warps.  n_nodes = the
 * number of rows / columns of A (while a bitmap of them fits in shared memory the columns are deduplicated per SM first). */
int kgat_frontier_expand(const int32_t* tasks, int64_t n_heavy_tasks, const int32_t* light_rank, const int32_t* col_idx,
                         const int32_t* rows, const int32_t* count_dev, int64_t max_rows, const uint32_t* level_bitmap,
                         uint8_t* flags, int64_t n_nodes, void* stream);
/* bitmap <- flags (every word written; flags cleared); rows[0 .. *count_dev) = ascending node ids of the set bits;
 * scratch: kgat_frontier_scratch_ints(n_nodes) int32 */
int64_t kgat_frontier_scratch_ints(int64_t n_nodes);
int kgat_frontier_list(uint8_t* flags, uint32_t* bitmap, int64_t n_nodes, int32_t* scratch, int32_t* rows, int32_t* count_dev,
                       void* stream);
/* The part of a level inside the node range [lo, hi) (lo a multiple of 32; hi a multiple of 32 or n_nodes): out_rows / out_count_dev
 * = that segment of the ascending row list, out_bitmap = the level's bitmap with every word outside the range cleared.
 * (Row-sharded runs: a rank computes the dense first layer for "level 1 AND my rows".) */
int kgat_frontier_segment(const int32_t* rows, const int32_t* count_dev, const uint32_t* bitmap, int64_t n_nodes, int64_t lo, int64_t hi,
                          int32_t* out_rows, int32_t* out_count_dev, uint32_t* out_bitmap, void* stream);
/* T[rows[i], 0:d] = 0 for i < *count_dev (gradient rows of the last table before the BPR scatter) */
int kgat_frontier_zero_rows(float* T, int64_t ld, int32_t d, const int32_t* rows, const int32_t* count_dev, int64_t max_rows,
                            void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K2/K3: bi-interaction aggregator   reference aggregator.py:57-65                              */
/* ------------------------------------------------------------------------------------------- */
/* out = normalize( dropout( lrelu((E+S) W1^T + b1) + lrelu((E*S) W2^T + b2) ) ), row-wise L2, eps 1e-12.
 * W1, W2: d_out x d_in row-major (nn.Linear.weight).  Dropout: p in [0,1); keep decisions come from
 * keep_bits (packed, (d_out+31)/32 words per row, bit=1 keeps) when non-NULL, else from the Philox
 * counter RNG (seed, offset) when p > 0; seed_dev (nullable device u64, e.g. the optimiser's step
 * counter) is mixed into the seed so a replayed CUDA graph draws a fresh mask every step.  Saved for backward: inv_norm[n] (1/max(||x||,eps); negative
 * when the eps clamp was active) and flags[n x d_out] (bit0: z1 > 0, bit1: z2 > 0, bit2: kept).
 * Row-sharded use: with n_peers > 0 the output rows are ALSO stored at the same row offset behind each of the
 * n_peers device pointers in the DEVICE array peer_out (the peers' copies of the table, kgat_peer_import), tile by
 * tile from the kernel's epilogue, so the exchange overlaps the computation; (NULL, 0) otherwise. */
int kgat_biagg_forward(const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out, const float* W1,
                       const float* b1, const float* W2, const float* b2, float dropout_p, uint64_t seed,
                       uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits, float* out, int64_t ld_out,
                       float* inv_norm, uint8_t* flags, float* const* peer_out, int32_t n_peers, void* stream);

/* Backward of the above.  g_out: n x d_out (ld_gout).  Produces g_S and g_E_direct (n x d_in) and
 * per-CTA partial parameter gradients in `partials` (n_ctas x (2*d_out*d_in + 2*d_out) floats,
 * n_ctas from kgat_biagg_backward_ctas), which kgat_biagg_reduce_param_grads sums in a fixed order
 * into gW1, gb1, gW2, gb2 (accumulate = 0 overwrites, 1 adds).  peer_gS / n_peers: as peer_out above, for g_S. */
int kgat_biagg_backward_ctas(int64_t n, int32_t d_in, int32_t d_out);
int kgat_biagg_backward(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm,
                        const uint8_t* flags, const float* E, const float* S, int64_t n, int32_t d_in, int32_t d_out,
                        const float* W1, const float* W2, float dropout_p, float* g_S, float* g_E, float* partials,
                        int32_t n_ctas, float* const* peer_gS, int32_t n_peers, void* stream);
int kgat_biagg_reduce_param_grads(const float* partials, int32_t n_ctas, int32_t d_in, int32_t d_out, float* gW1,
                                  float* gb1, float* gW2, float* gb2, int32_t accumulate, void* stream);

/* Forward / backward over a needed-row list (frontier section): the kernels process the *n_rows_dev rows listed in
 * row_ids (max_rows = capacity of the list, sizes the grid); every per-row array (E, S, out, inv_norm, flags,
 * keep_bits, g_out, g_S, g_E, the dropout stream) stays indexed by NODE id, rows outside the list are not touched. */
int kgat_biagg_forward_rows(const float* E, const float* S, const int32_t* row_ids, const int32_t* n_rows_dev, int64_t max_rows,
                            int32_t d_in, int32_t d_out, const float* W1, const float* b1, const float* W2, const float* b2,
                            float dropout_p, uint64_t seed, uint64_t offset, const uint64_t* seed_dev, const uint32_t* keep_bits,
                            float* out, int64_t ld_out, float* inv_norm, uint8_t* flags, void* stream);
int kgat_biagg_backward_rows_ctas(int64_t max_rows, int32_t d_in, int32_t d_out);
int kgat_biagg_backward_rows(const float* g_out, int64_t ld_gout, const float* out, int64_t ld_out, const float* inv_norm,
                             const uint8_t* flags, const float* E, const float* S, const int32_t* row_ids,
                             const int32_t* n_rows_dev, int64_t max_rows, int32_t d_in, int32_t d_out, const float* W1,
                             const float* W2, float dropout_p, float* g_S, float* g_E, float* partials, int32_t n_ctas,
                             void* stream);

/* T[ids64[i], 0:d] = 0 (ids outside [0, n_rows) ignored): re-zero the rows a batch's gradient scatter touched instead of
 * clearing a whole n_rows x d gradient table per step (model.py:211-261 touches <= 3B of the N embedding rows) */
int kgat_zero_rows_i64(float* T, int64_t n_rows, int64_t ld, int32_t d, const int64_t* ids64, int64_t n_ids, void* stream);

/* Dense view of the compact TransR gradient rows (kgat_transr_step): dense[id, :] = g_rows[row_slot[id], :] for the batch's
 * ids -- what autograd hands out as embedding.weight.grad (model.py:204-261), zero outside those rows, kept valid by
 * kgat_transr_release_rows(previous batch's ids) = clear those rows and free their row_slot claims. */
int kgat_transr_rows_to_dense(const float* g_rows, const int32_t* row_slot, const int64_t* heads, const int64_t* pos_tails,
                              const int64_t* neg_tails, int32_t batch, int32_t d, float* dense, int64_t ld, int64_t* keep_heads,
                              int64_t* keep_pos_tails, int64_t* keep_neg_tails /* optional: copies of the ids, all three or none */,
                              void* stream);
int kgat_transr_release_rows(float* dense, int64_t n_rows, int64_t ld, int32_t d, const int64_t* ids64, int64_t n_ids,
                             int32_t* row_slot, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K4: BPR loss over the layer tables      reference model.py:189-202, 142-163                   */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_tables;
    int32_t dims[KGAT_MAX_LAYERS];
    const float* tables[KGAT_MAX_LAYERS]; /* table l: n_nodes x dims[l] */
    int64_t lds[KGAT_MAX_LAYERS];
} kgat_tables_t;

typedef struct {
    int32_t n_tables;
    int32_t dims[KGAT_MAX_LAYERS];
    float* tables[KGAT_MAX_LAYERS];
    int64_t lds[KGAT_MAX_LAYERS];
} kgat_grad_tables_t;

/* Optional publication of a step's loss to the host by the kernel that reduces it (what kgat_publish_loss does as a launch of
 * its own): ring_host_mapped[s % n_slots] = (s << 32) | float bits of the loss, with s = ++serial_dev[0]; the ring lives in
 * mapped pinned host memory, so loss.item() is a host-side poll that does not wait for the kernels queued behind the loss. */
typedef struct {
    uint64_t* serial_dev;
    uint64_t* ring_host_mapped;
    int32_t n_slots;
} kgat_publish_t;

/* loss[0] = -mean(logsigmoid(pos - neg)) + reg * (mean|u|^2/2 + mean|p|^2/2 + mean|n|^2/2);
 * margin: scratch of 2*batch floats: [pos_b - neg_b (saved for the backward)][per-sample l2 term].
 * ids are used as given (no user offset, SURVEY.md Q4).  loss_sum (may be NULL): loss_sum[0] += loss[0] in the same launch. */
int kgat_bpr_forward(const kgat_tables_t* tables, const int64_t* users, const int64_t* pos, const int64_t* neg,
                     int32_t batch, float reg, float* loss, float* loss_sum, float* margin, const kgat_publish_t* publish /* may be NULL */,
                     void* stream);
/* Scatter-adds d loss / d table rows into grad tables (atomicAdd; tables[l] may be NULL to skip a
 * layer).  g_loss: device scalar (upstream gradient). */
int kgat_bpr_backward(const kgat_tables_t* tables, const kgat_grad_tables_t* grads, const int64_t* users,
                      const int64_t* pos, const int64_t* neg, int32_t batch, float reg, const float* margin,
                      const float* g_loss, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K5: TransR loss                           reference model.py:204-261                          */
/* ------------------------------------------------------------------------------------------- */
/* emb: n_nodes x d; rel_emb: n_rel x k; W: n_rel x d x k (row-vector convention x = e W_r).
 * loss[0] = -mean(logsigmoid(neg - pos)) + reg * (4 l2 means).  No W_r materialisation. */
int kgat_transr_forward(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k,
                        const int64_t* heads, const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails,
                        int32_t batch, float reg, float* loss, float* margin, void* stream);
/* Accumulates (atomicAdd) into g_emb (n_nodes x d), g_rel_emb (n_rel x k), g_W (n_rel x d x k);
 * the caller zeroes them.  With row_slot != NULL, g_emb is instead a compact 3*batch x d buffer and node i
 * accumulates into row row_slot[i] (kgat_transr_claim_rows). */
int kgat_transr_backward(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k,
                         const int64_t* heads, const int64_t* rels, const int64_t* pos_tails,
                         const int64_t* neg_tails, int32_t batch, float reg, const float* margin, const float* g_loss,
                         float* g_emb, float* g_rel_emb, float* g_W,
                         const int32_t* row_slot, void* stream);
/* The whole TransR part of a KG training step in three launches (model.py:204-261 forward + its autograd backward):
 * (1) claim compact gradient rows (kgat_transr_claim_rows) and zero g_rows, g_rel_emb (n_rel x k), g_W in the same
 * launch; (2) forward and backward in one pass -- the backward recomputes the projections anyway -- with
 * d loss = 1, gradients into g_rows (through row_slot), g_rel_emb, g_W; (3) loss[0] = batch loss, and
 * loss_sum[0] += loss[0] when loss_sum != NULL.  margin: 2 * batch floats of scratch. */
int kgat_transr_step(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, int32_t n_rel,
                     const int64_t* heads, const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch,
                     float reg, float* loss, float* loss_sum, float* margin, int32_t* row_slot, float* g_rows, float* g_rel_emb,
                     float* g_W, const kgat_publish_t* publish /* may be NULL */, void* stream);
/* One slot per distinct node of a TransR batch: row_slot (n_nodes int32, -1 = free) gets, for every node among
 * heads / pos_tails / neg_tails, the index in [0, 3*batch) of its first claimant; g_rows (3*batch x d) is zeroed.
 * kgat_adam_apply (row_slot0) consumes the rows and frees the slots. */
int kgat_transr_claim_rows(const int64_t* heads, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, int32_t d,
                           int32_t* row_slot, float* g_rows, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K6-K8: attention refresh                  reference model.py:263-366,                         */
/*                                           multi_head_attention.py:35-58                       */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    const float* Wv; /* d x d  _value_weight.weight (out x in) */
    const float* bv;
    const float* Wo; /* d x d  _output.weight */
    const float* bo;
    const float* ln_gamma;
    const float* ln_beta;
    float ln_eps;
    int32_t n_heads;
} kgat_mha_t;

/* MultiHeadAttention.forward (multi_head_attention.py:35-58) on caller-provided projected tail embeddings (n x d):
 * out = LayerNorm(Wo drop(Wv x + bv) + bo), n x d.  The query / key inputs cancel (softmax over a length-1 axis,
 * SURVEY.md Q1) and are not taken.  Per-head dropout as in kgat_att_edge_scores_dropout (head_bits: one byte per row,
 * bit h keeps head h; else Philox (seed, offset + row)); dropout_p = 0 in eval mode. */
int kgat_mha_forward(const float* tail_embedding, int64_t n, int32_t d, const kgat_mha_t* mha, float dropout_p,
                     const uint8_t* head_bits, uint64_t seed, uint64_t offset, float* out, void* stream);

/* Canonical KGAT score (north_star (1); the paper's pi(h, r, t) = (W_r e_t)^T tanh(W_r e_h + e_r), row-vector convention
 * x = e W_r of model.py:291-298) -- an OPTION (model.score_mode = "kgat"); the reference itself scores edges with the value path
 * of its multi-head attention (below).  x_out[p] = emb[pair_node[p]] W[pair_rel[p]] for unique (node, relation) pairs, then
 * score[e] = sum_j x_tail[tail_pair[e]][j] * tanh(x_head[head_pair[e]][j] + rel_emb[edge_rel[e]][j]). */
int kgat_att_pair_project(const float* emb, const float* W, int32_t d, const int32_t* pair_node, const int32_t* pair_rel,
                          int64_t n_pairs, float* x_out, void* stream);
int kgat_att_edge_scores_kgat(const float* x_head, const int32_t* head_pair, const float* x_tail, const int32_t* tail_pair,
                              const float* rel_emb, const int32_t* edge_rel, int64_t n_edges, int32_t d, float* score_out,
                              void* stream);

/* Per unique (tail, relation) pair: x = e_t W_r, v = Wv x + bv.  If v_out != NULL stores v (n_pairs x d).
 * If score_out != NULL also o = Wo v + bo, LayerNorm, score = sum tanh  (the eval-mode edge score
 * before the degree weight: the reference's query/key path cancels, SURVEY.md Q1). d = k = 64. */
int kgat_att_pair_scores(const float* emb, const float* W, int32_t d, const int32_t* pair_tail,
                         const int32_t* pair_rel, int64_t n_pairs, const kgat_mha_t* mha, float* v_out,
                         float* score_out, void* stream);
/* Train-mode (attention dropout live, SURVEY.md Q2): per edge, per-head keep decision from head_bits
 * (one byte per edge, bit h keeps head h) when non-NULL else from Philox(seed, offset + edge);
 * kept heads are scaled by 1/(1-p).  score[e] = sum tanh(LN(Wo (mask * v[pair_of_edge[e]]) + bo)). */
int kgat_att_edge_scores_dropout(const float* pair_v, const int32_t* pair_of_edge, int64_t n_edges, int32_t d,
                                 const kgat_mha_t* mha, float dropout_p, const uint8_t* head_bits, uint64_t seed,
                                 uint64_t offset, const uint64_t* seed_dev, float* score_out, void* stream);
/* Row softmax over CSR slots with duplicate merge.  Edges are given in slot-sorted order: slot s owns
 * sorted edges [slot_ptr[s], slot_ptr[s+1]).  Edge score = (pair_score ? pair_score[pair_of_edge[p]] :
 * edge_score[p]) * edge_weight[p].  vals[s] = softmax over the row of sum of its edges' scores. */
int kgat_att_row_softmax(const int32_t* row_ptr, int64_t n_rows, const int32_t* slot_ptr, const float* pair_score,
                         const int32_t* pair_of_edge, const float* edge_score, const float* edge_weight, float* vals,
                         void* stream);
/* edge_weight[p] = mult / (log1p(deg_h) + log1p(deg_t))     reference model.py:309-314 */
int kgat_att_edge_weights(const int32_t* deg_head, const int32_t* deg_tail, const float* mult, int64_t n_edges,
                          float* edge_weight, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K9/K10: predict                           reference model.py:388-391, metrics_calculator.py   */
/* ------------------------------------------------------------------------------------------- */
/* out[b, :] = concat_l tables[l][ids[b], :]   (b < n_ids; out: n_ids x sum(dims), ld_out) */
int kgat_gather_concat(const kgat_tables_t* tables, const int64_t* ids64, int64_t n_ids, float* out, int64_t ld_out,
                       void* stream);
/* C (m x n) = A (m x k) * B^T (n x k), fp32 CUDA cores with fp32 accumulation */
int kgat_sgemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int32_t m,
                  int32_t n, int32_t k, void* stream);
/* In-place mask: scores[b, items of user b] = -inf  (CSR-like mask_ptr / mask_items, int32) */
int kgat_mask_scores(float* scores, int64_t ld, int32_t m, int32_t n, const int32_t* mask_ptr,
                     const int32_t* mask_items, void* stream);
/* Top-K per row, descending, exact ties broken lowest column first (CPU torch.sort order).
 * k <= 128.  idx_out: m x k int32, val_out (optional): m x k. */
int kgat_topk_rows(const float* scores, int64_t ld, int32_t m, int32_t n, int32_t k, int32_t* idx_out,
                   float* val_out, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Path explanations: why a problem reaches a user through A (no counterpart in the reference,     */
/* whose --visualize_attention / weights_visualizer.py:19 read single entries attentive_matrix[u,p]) */
/* ------------------------------------------------------------------------------------------- */
/* For each of n_pairs pairs (src[j], dst[j]) of node ids (int32, e.g. from kgat_ids64_to_i32): the simple paths
 * s = v0 -> v1 -> ... -> vh = t of 1 <= h <= max_hops (max_hops in {1, 2, 3}) hops whose every hop (v_m, v_m+1) is a
 * stored entry of A (a column of CSR row v_m; the direction of propagation, so the path carries t's embedding into s).
 * Weight = fp32 product of the hop values left to right, ((A[v0,v1] * A[v1,v2]) * A[v2,v3]).  Paths rank by weight
 * descending, then h ascending, then (v1, v2) ascending.  s == t, or an id outside [0, n_nodes), has no paths.
 * A: CSR (row_ptr, col_idx, vals) with sorted unique columns per row, and its transpose (t_ptr, t_idx) with t_perm mapping
 * a transposed slot to its CSR slot (graph.py: AttentiveGraph).  k in [1, 64].  Outputs (P = n_pairs, H = max_hops):
 *   nodes  int64 [P, k, H+1]  v0..vh, -1 after vh and for missing paths
 *   slots  int64 [P, k, H]    CSR slot of every hop (= index into the COO view's indices / values), -1 padding
 *   hops   int32 [P, k]       h, 0 for a missing path
 *   weight fp32  [P, k]       path weight, 0 for a missing path
 *   count  int64 [P, H]       number of simple paths of each length
 *   mass   fp32  [P, H]       their summed weight (fp64 sums in a fixed order: bitwise reproducible)
 * Work per pair is sum over the intersections (row s & In t, row a & In t for a in row s) of the shorter list times
 * log of the longer; it is spread over several CTAs per pair.  Two launches, no host synchronisation; workspace
 * size from kgat_explain_paths_workspace_bytes (depends on n_pairs and k only; -1 for invalid arguments). */
int64_t kgat_explain_paths_workspace_bytes(int64_t n_pairs, int32_t k, int32_t max_hops);
int kgat_explain_paths(const int32_t* row_ptr, const int32_t* col_idx, const float* vals, const int32_t* t_ptr, const int32_t* t_idx,
                       const int32_t* t_perm, int64_t n_nodes, const int32_t* src, const int32_t* dst, int64_t n_pairs, int32_t k,
                       int32_t max_hops, int64_t* nodes, int64_t* slots, int32_t* hops, float* weight, int64_t* count, float* mass,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Filtered top-k recommendations for many users in one call (the reference's recommend(),        */
/* main.py:541-636, loops over 256-user batches of a materialised score matrix)                   */
/* ------------------------------------------------------------------------------------------- */
/* Candidate filter.  Item items[i] (int32, in [0, n_nodes - user_num)) passes iff, for every group g < n_groups, CSR row
 * user_num + items[i] of A (sorted unique columns) stores a column among group_nodes[group_ptr[g] .. group_ptr[g+1]) (node
 * ids; a stored entry counts whatever its value).  n_groups = 0 passes every item.  Outputs, in input order: positions[j] =
 * index into items of the j-th passing item, cand_items[j] = items[positions[j]] (both n_items int32; `positions` is also
 * the scratch of the flags), *n_cand = their number (device int32).  Two launches, no host synchronisation. */
int kgat_recommend_filter(const int32_t* row_ptr, const int32_t* col_idx, int64_t n_nodes, int32_t user_num, const int32_t* items,
                          int64_t n_items, const int32_t* group_ptr, const int32_t* group_nodes, int32_t n_groups, int32_t* positions,
                          int32_t* cand_items, int32_t* n_cand, void* stream);
/* Top-k candidates per user without materialising scores.  users[b]: table rows (int32); candidates: cand_items[0 .. n)
 * (int32 table rows, unique), n = *n_cand when n_cand != NULL (e.g. from kgat_recommend_filter) else n_cand_max.
 * Score(b, c) = sequential fp32 fmaf chain over the concatenated row of the tables from +0 (zero columns padded to a multiple
 * of 16), exactly kgat_gather_concat + kgat_sgemm_nt.  exclude_ptr / exclude_items (nullable): CSR over table rows of users,
 * items ascending per user; candidate c is skipped for user b when cand_items[c] is in users[b]'s list.  Order: descending
 * key of kgat_topk_rows (NaN largest, -0 below +0), then lower candidate index.  k in [1, 128]; slices in [0, 64] = candidate
 * slices per 64-user tile (0 = chosen from n_users, the SM count and the CTAs per SM; the result does not depend on it).  Outputs:
 *   out_items  int64 [n_users, k]  cand_items of the ranked candidates, -1 after out_count[b]
 *   out_scores fp32  [n_users, k]  their scores, -inf after out_count[b]
 *   out_count  int32 [n_users]     min(k, number of candidates not excluded for users[b])
 * Two launches, no host synchronisation; workspace from kgat_recommend_workspace_bytes with the same arguments (-1 for
 * invalid ones, or a row too wide for shared memory).  KGAT_ERR_UNSUPPORTED when the concatenated row is too wide for shared
 * memory at this k. */
int64_t kgat_recommend_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_cand_max, int32_t k, int32_t slices);
int kgat_recommend_topk(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand_max,
                        const int32_t* n_cand, int32_t k, const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices,
                        int64_t* out_items, float* out_scores, int32_t* out_count, void* workspace, int64_t workspace_bytes, void* stream);
/* Top-k with per-group caps (a varied practice set: at most c_j problems of group j).  Group masks first: for candidate
 * c < n (n as for kgat_recommend_topk), bit g of masks[4 c + g / 32] (bit g % 32) is set iff CSR row user_num + cand_items[c]
 * of A stores a column among group_nodes[group_ptr[g] .. group_ptr[g+1]) -- the membership test of kgat_recommend_filter.
 * n_groups in [0, 128]; masks uint32 [n_cand_max, 4].  One launch, no host synchronisation. */
int kgat_recommend_group_masks(const int32_t* row_ptr, const int32_t* col_idx, int64_t n_nodes, int32_t user_num, const int32_t* cand_items,
                               int64_t n_cand_max, const int32_t* n_cand, const int32_t* group_ptr, const int32_t* group_nodes, int32_t n_groups,
                               uint32_t* masks, void* stream);
/* Then rounds r = 0, 1, ... of the exact greedy: for row b, walk its eligible candidates (as for kgat_recommend_topk) in
 * kgat_recommend_topk's order and accept c when every group g of c has count_g < caps[g] (int32 [n_groups], each >= 0);
 * accepting adds 1 to count_g for each group of c; stop at k acceptances.  Round r takes, for each
 * of its n_active rows, the top m (k <= m <= 128) candidates after the row's last entry of round r - 1 that touch no group
 * already at its cap, and walks them.  A row is finished when it has k entries or the round found fewer than m; the others
 * go to round r + 1, *n_active_next of them (device int32, written by the call).  Round 0 takes n_active = n_users; call
 * the next round with the value read back from *n_active_next until it is 0, with the same arguments and workspace
 * otherwise.  At most n_groups + 1 rounds.  Outputs, complete once no row is active:
 *   out_items  int64 [n_users, k]  cand_items of the accepted candidates in acceptance order, -1 after out_count[b]
 *   out_scores fp32  [n_users, k]  their scores (bit-identical to kgat_recommend_topk), -inf after out_count[b]
 *   out_count  int32 [n_users]     number of accepted candidates
 * slices in [0, 64] (0 = the rule of kgat_recommend_topk, applied to each round's active rows; the result does not depend
 * on it).  Two launches per round, no host synchronisation; workspace from kgat_recommend_capped_workspace_bytes with the
 * same arguments (-1 for invalid ones, or a row too wide for shared memory at m, when the round returns KGAT_ERR_UNSUPPORTED). */
int64_t kgat_recommend_capped_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_cand_max, int32_t n_groups, int32_t k,
                                              int32_t m, int32_t slices);
int kgat_recommend_capped_round(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand_max,
                                const int32_t* n_cand, const uint32_t* masks, const int32_t* caps, int32_t n_groups, int32_t k, int32_t m,
                                const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices, int32_t round, int64_t n_active,
                                int32_t* n_active_next, int64_t* out_items, float* out_scores, int32_t* out_count, void* workspace,
                                int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Exact full ranking of held-out targets (the full-ranking metrics: rank, MRR, AUC, any k)      */
/* ------------------------------------------------------------------------------------------- */
/* For every users[b] (int32 table row) and each of its targets p = target_items[target_ptr[u] .. target_ptr[u+1]) (ascending,
 * table rows), the exact number of eligible candidates that outrank p.  Candidates: cand_items[0 .. n_cand) (int32 table rows,
 * unique); the position of an item is given by pos_map[item] (int32 [n_pos], -1 when not a candidate) or, when pos_map is
 * NULL, by the item itself (then cand_items[c] must be c).  exclude_ptr / exclude_items (nullable): CSR over table rows of
 * users, items ascending; an excluded item is not eligible.  Score s(b, c) as in kgat_recommend_topk; key K(b, c) =
 * (topk_rows key of s << 32) | (0xFFFFFFFF - position of c), the order of kgat_recommend_topk.  Outputs, row b at
 * out_ptr[b] .. out_ptr[b+1] (int64 [n_users + 1], out_ptr[b+1] - out_ptr[b] = number of targets of users[b],
 * out_ptr[n_users] = n_targets):
 *   out_items    int64 [n_targets]  the targets, ascending
 *   out_scores   fp32  [n_targets]  s(b, p), bit-identical to kgat_gather_concat + kgat_sgemm_nt
 *   out_rank     int64 [n_targets]  #{eligible c : K(b, c) > K(b, p)}, or -1 when p is not eligible
 *   out_eligible int64 [n_users]    number of eligible candidates of users[b]
 * slices in [0, 64] = candidate slices per 64-user tile (0 = the rule of kgat_recommend_topk; the result does not depend on
 * it).  Three launches, no host synchronisation; workspace from kgat_rank_workspace_bytes (-1 for invalid arguments or a row
 * too wide for shared memory, when kgat_rank_targets returns KGAT_ERR_UNSUPPORTED). */
int64_t kgat_rank_workspace_bytes(const kgat_tables_t* tables, int64_t n_users, int64_t n_targets);
int kgat_rank_targets(const kgat_tables_t* tables, const int32_t* users, int64_t n_users, const int32_t* cand_items, int64_t n_cand,
                      const int32_t* pos_map, int64_t n_pos, const int32_t* target_ptr, const int32_t* target_items, const int64_t* out_ptr,
                      int64_t n_targets, const int32_t* exclude_ptr, const int32_t* exclude_items, int32_t slices, int64_t* out_items,
                      float* out_scores, int64_t* out_rank, int64_t* out_eligible, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Knowledge-graph completion with the trained TransR half: top-k tails and filtered ranks       */
/* ------------------------------------------------------------------------------------------- */
/* Queries (h, r) = (heads[q], rels[q]) (int32 CKG node / relation ids), sorted by relation: segment g holds the queries
 * seg_ptr_host[g] .. seg_ptr_host[g+1] (host int64 [n_seg + 1], each segment non-empty) of relation seg_rel[g] (device int32
 * [n_seg]); row q_out[q] of the outputs belongs to query q.  emb [n_nodes, d], rel_emb [n_rel, kdim], W [n_rel, d, kdim]: the
 * TransR parameters, d = kdim in {32, 64, 128} (KGAT_ERR_UNSUPPORTED otherwise).
 * Energy E(h, r, t) = ||e_h W_r + e_r - e_t W_r||^2 in fp32, bit-identical to the per-sample term of kgat_transr_forward
 * (margin = E(h, r, n) - E(h, r, p)).  Key K(q, c) = (float_key(-E) << 32) | (0xFFFFFFFF - c), c = position in cand (int32
 * node ids, unique); a NaN energy keys as the largest value (ranks first).  ex_keys (nullable): ascending int64 keys
 * (h n_rel + r) n_nodes + t of known triples; candidate c is not eligible for (h, r) when (h, r, cand[c]) is known.
 * slices in [0, 64]: candidate slices per 64-query tile (0 = the rule of kgat_recommend_topk; the result does not depend
 * on it).  Candidate projections are computed for up to 32 relations at a time, within 1 GiB.  Workspace from
 * kgat_complete_workspace_bytes(d, kdim, n_q, n_tiles, n_cand, n_seg, k, slices, count) with n_tiles = sum over segments of
 * ceil(size / 64) and count = 1 for kgat_complete_rank (k ignored), 0 for kgat_complete_topk; -1 for invalid arguments.
 * No host synchronisation. */
int64_t kgat_complete_workspace_bytes(int32_t d, int32_t kdim, int64_t n_queries, int64_t n_tiles, int64_t n_cand, int32_t n_rel_used, int32_t k,
                                      int32_t slices, int32_t count);
/* Top-k eligible tails per query, lowest energy first: out_tails int64 [n_q, k] (node ids, -1 after out_count[row]),
 * out_energy fp32 [n_q, k] (+inf after out_count[row]), out_count int32 [n_q] = min(k, eligible candidates); k in [1, 128]. */
int kgat_complete_topk(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t kdim, int64_t n_nodes, int64_t n_rel,
                       const int32_t* heads, const int32_t* rels, const int32_t* q_out, int64_t n_q, const int64_t* seg_ptr_host,
                       const int32_t* seg_rel, int32_t n_seg, const int32_t* cand, int64_t n_cand, const int64_t* ex_keys, int64_t n_ex,
                       int32_t k, int32_t slices, int64_t* out_tails, float* out_energy, int32_t* out_count, void* workspace,
                       int64_t workspace_bytes, void* stream);
/* Filtered rank of the target tails[q]: out_rank int64 [n_q] = #{eligible c != t : K(q, c) > K(q, t)} (the target stays
 * eligible even when (h, r, t) is known), -1 when t is not a candidate; out_energy fp32 [n_q] = E(h, r, t); out_eligible int64
 * [n_q] = candidates not known for (h, r), the target counted.  pos_map (nullable): int32 [n_nodes], position of a node in
 * cand or -1; NULL means cand[c] == c. */
int kgat_complete_rank(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t kdim, int64_t n_nodes, int64_t n_rel,
                       const int32_t* heads, const int32_t* rels, const int32_t* tails, const int32_t* q_out, int64_t n_q,
                       const int64_t* seg_ptr_host, const int32_t* seg_rel, int32_t n_seg, const int32_t* cand, int64_t n_cand,
                       const int32_t* pos_map, const int64_t* ex_keys, int64_t n_ex, int32_t slices, float* out_energy, int64_t* out_rank,
                       int64_t* out_eligible, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* K11: Adam                               reference model.py:393-419 (torch.optim.Adam)       */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_tensors;
    float* param[KGAT_MAX_TENSORS];
    const float* grad[KGAT_MAX_TENSORS];
    float* exp_avg[KGAT_MAX_TENSORS];
    float* exp_avg_sq[KGAT_MAX_TENSORS];
    int64_t numel[KGAT_MAX_TENSORS];
    /* row-sharded use: the updated values of tensor 0 (this rank's embedding rows) are also stored at the same
     * offset behind each of the n_peers device pointers of the DEVICE array peer_param0; (NULL, 0) otherwise */
    float* const* peer_param0;
    int32_t n_peers;
    /* row-sparse gradient for tensor 0 (the embedding table in the KG phase): when row_slot0 != NULL, grad[0] holds
     * compact rows [n_slots x row_dim0] and row r of tensor 0 uses row row_slot0[r] of it (g = 0 where the slot is
     * -1); the kernel resets the used slots to -1.  See kgat_transr_claim_rows. */
    int32_t* row_slot0;
    int32_t row_dim0;
} kgat_adam_tensors_t;
/* One torch.optim.Adam step (no weight decay, no amsgrad) over all listed tensors in one launch,
 * split in two so a captured CUDA graph replays correctly: kgat_adam_advance increments the device
 * step counter and writes the step-dependent scalars {1-b1, b2, 1-b2, lr/bc1, 1/sqrt(bc2), eps} to
 * hyper_dev (6 floats, bias corrections in double); kgat_adam_apply streams over the tensors. */
int kgat_adam_advance(int64_t* step_dev, double lr, double beta1, double beta2, double eps, float* hyper_dev, void* stream);
/* same scalars from a host-known 1-based step (the torch.optim.Optimizer path keeps step on the host) */
int kgat_adam_set_hyper(int64_t step, double lr, double beta1, double beta2, double eps, float* hyper_dev, void* stream);
int kgat_adam_apply(const kgat_adam_tensors_t* t, const float* hyper_dev, void* stream);

/* Lazy but exact Adam for a row-sparse phase (the KG phase: a TransR batch touches <= 3B of the N embedding
 * rows, while torch.optim.Adam sweeps all N rows every step, model.py:414-419).  Each row carries the number
 * of phase steps it is current to (row_step, int32, 0 at phase start = optimiser step s0, a device scalar so
 * that captured graphs survive across phases).  A row is caught
 * up -- the zero-gradient update replayed step by step with each step's own bias corrections from
 * `table` ({lr/bc1_s, 1/sqrt(bc2_s)} for s = s0+1 .. s0+n_steps) -- when a batch is about to read it
 * (catchup, before the forward; cur_step_dev = steps done), gets its real gradient after the backward
 * (sparse_rows, after kgat_adam_advance; the gradient row is re-zeroed), and all rows are caught up at the
 * end of the phase (flush).  Bit-identical to the dense sweep.  hyper_dev as written by kgat_adam_advance. */
int kgat_adam_hyper_table(const int64_t* s0_dev, int32_t n_steps, double lr, double beta1, double beta2, float* table, void* stream);
int kgat_adam_lazy_catchup(float* param, float* exp_avg, float* exp_avg_sq, int32_t* row_step, const int64_t* ids, int32_t n_ids,
                           int32_t d, const int64_t* cur_step_dev, const int64_t* s0_dev, const float* table, const float* hyper_dev, void* stream);
int kgat_adam_sparse_rows(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int32_t* row_step, const int64_t* ids,
                          int32_t n_ids, int32_t d, const int64_t* cur_step_dev, const int64_t* s0_dev, const float* hyper_dev, void* stream);
int kgat_adam_lazy_flush(float* param, float* exp_avg, float* exp_avg_sq, int32_t* row_step, int64_t n_rows, int32_t d,
                         const int64_t* cur_step_dev, const int64_t* s0_dev, const float* table, const float* hyper_dev, void* stream);

/* Rolling-window exact Adam for the KG phase (the epoch engine's default; replaces the per-step dense sweep of
 * torch.optim.Adam over the N x d embedding table, model.py:414-419, with bit-identical results).  The table is cut
 * into `window` contiguous slices; phase step j replays the zero-gradient updates of slice (j - 1) mod window up to
 * step j - 1, so no row lags more than window + 1 steps and a step moves 1/window of the optimiser state through HBM.
 *   kgat_adam_rolling_prepare  before the forward: claims the batch's compact gradient rows (as kgat_transr_claim_rows),
 *                              zeroes g_rows and the two optional buffers zero_a / zero_b (n_a / n_b floats, multiples of
 *                              4), and brings every batch row up to the steps done so far (cur_step_dev - s0_dev);
 *   kgat_transr_step_claimed   kgat_transr_step minus its claim launch;
 *   kgat_adam_rolling_apply    after kgat_adam_advance: claimed rows take their gradient (step j) and free their slot,
 *                              the tensors of `dense` (may be NULL) take a plain Adam step, the slice is replayed;
 *   kgat_adam_lazy_flush       end of the phase.
 * row_step / s0_dev / table / hyper_dev as for the lazy scheme above.  `advanced` = 1 when the step counter was already
 * advanced for this step (kgat_step_begin_i64), so the steps done are one fewer.  `parts`: bit 0 = claimed rows + dense tensors,
 * bit 1 = slice replay; the two parts touch disjoint rows (ownership through atomicMax on row_step) and may run as concurrent
 * launches on two streams once the prepare launch has finished.  dense (may be NULL) + prev_*: the API path's dense view of
 * the embedding gradient (kgat_transr_rows_to_dense) still holds the previous batch's rows; the prepare launch clears them. */
int kgat_adam_rolling_prepare(const int64_t* heads, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, int32_t d,
                              int32_t* row_slot, float* g_rows, float* zero_a, int64_t n_a, float* zero_b, int64_t n_b, float* param,
                              float* exp_avg, float* exp_avg_sq, int32_t* row_step, const int64_t* cur_step_dev, int32_t advanced,
                              const int64_t* s0_dev, const float* table, const float* hyper_dev, const int64_t* prev_heads,
                              const int64_t* prev_pos_tails, const int64_t* prev_neg_tails, float* dense, int64_t ld_dense, void* stream);
int kgat_transr_step_claimed(const float* emb, const float* rel_emb, const float* W, int32_t d, int32_t k, const int64_t* heads,
                             const int64_t* rels, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, float reg, float* loss,
                             float* loss_sum, float* margin, const int32_t* row_slot, float* g_rows, float* g_rel_emb, float* g_W,
                             const kgat_publish_t* publish /* may be NULL */, void* stream);
int kgat_adam_rolling_apply(const int64_t* heads, const int64_t* pos_tails, const int64_t* neg_tails, int32_t batch, int32_t d,
                            int32_t* row_slot, const float* g_rows, float* param, float* exp_avg, float* exp_avg_sq, int32_t* row_step,
                            int64_t n_rows, int32_t window, const kgat_adam_tensors_t* dense, int32_t parts, const int64_t* cur_step_dev,
                            const int64_t* s0_dev, const float* table, const float* hyper_dev, void* stream);

/* Device self-test of the Adam arithmetic core: for i < n computes q = m[i] / (sqrt(v[i]) * inv_sqrt_bc2 + eps) by the kernels'
 * branch-free sequences (with their fallback) and by the IEEE builtins; counts[0] += results whose bits differ, counts[1] +=
 * elements that stayed on the fast sequences.  counts: 2 int32, zeroed by the caller. */
int kgat_selftest_adam_arith(const float* m, const float* v, int64_t n, float inv_sqrt_bc2, float eps, int32_t* counts, void* stream);

/* dst[0..elems) = src[(counter_dev[0] % n_batches) * elems + ...]: selects the current step's pre-sampled
 * id batch from a device-resident epoch array (counter = an optimiser step counter) so that a captured
 * CUDA graph of a training step replays through the whole epoch without host work. */
int kgat_select_batch_i64(const int64_t* src, int64_t n_batches, int64_t elems, const int64_t* counter_dev, int64_t* dst,
                          void* stream);
/* kgat_select_batch_i64 followed by kgat_adam_advance on the same counter, in one single-CTA launch: the batch of step
 * counter % n_batches is selected, then the counter is incremented and hyper_dev written for the new step. */
int kgat_step_begin_i64(const int64_t* src, int64_t n_batches, int64_t elems, int64_t* step_dev, int64_t* dst, double lr, double beta1,
                        double beta2, double eps, float* hyper_dev, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* P5: batch samplers on the device       reference preprocess.py:328-415 (CF), 417-530 (KG)   */
/* ------------------------------------------------------------------------------------------- */
/* CF batch: `batch` distinct users out of active_users (with replacement only if batch > n_active), one uniform
 * positive item of the user, one uniform item not among the user's items (rejection, items sorted per user).
 * out = [users | pos | neg], 3 x batch int64.  Randomness = Philox(seed, step_dev[0], sample index). */
int kgat_sample_cf_batch(const int32_t* user_ptr, const int32_t* user_items, const int32_t* active_users, int32_t n_active,
                         int32_t item_num, int32_t batch, uint64_t seed, const int64_t* step_dev, int64_t* out, void* stream);
/* KG batch: `batch` distinct heads, one uniform (relation, tail) edge of the head, one uniform node that is not a
 * tail of (head, relation) (edges sorted by (head, tail)).  out = [heads | rels | pos tails | neg tails], 4 x batch. */
int kgat_sample_kg_batch(const int32_t* head_ptr, const int32_t* edge_rel, const int32_t* edge_tail, const int32_t* active_heads,
                         int32_t n_active, int32_t node_num, int32_t batch, uint64_t seed, const int64_t* step_dev, int64_t* out,
                         void* stream);

/* ------------------------------------------------------------------------------------------- */
/* (e) multi-GPU: row exchange over NVLink peer memory.  No counterpart in the reference (single   */
/* device); replaces the all-gather that follows every propagation layer of the row-sharded       */
/* aggregator.py:54-65 / its backward.  See csrc/peer.cu for the protocol.                        */
/* ------------------------------------------------------------------------------------------- */
/* The only entry points that allocate: an IPC-exportable, zero-filled device allocation, its 64-byte handle,
 * and the mapping of a peer's handle into this process (same node, NVLink / PCIe peer access). */
int kgat_peer_alloc(int64_t bytes, void** ptr);
int kgat_peer_free(void* ptr);
int kgat_peer_export(const void* ptr, void* handle64);
int kgat_peer_import(const void* handle64, void** ptr);
int kgat_peer_close(void* ptr);
/* Copy n_floats (multiple of 4, 16-byte aligned) from src to peer_dst[q] for q < n_peers.  peer_dst is a DEVICE
 * array of n_peers device pointers into the peers' mapped allocations.  max_ctas > 0 bounds the grid (a push that
 * runs beside compute kernels on another stream needs few SMs to fill the links); 0 = 8 CTAs per SM. */
int kgat_peer_push(const float* src, float* const* peer_dst, int32_t n_peers, int64_t n_floats, int32_t max_ctas, void* stream);
/* The *count_dev rows listed in `rows` (node ids) of `table` (row stride ld floats) -> the same rows of every peer's table
 * (DEVICE array of n_peers base pointers).  The row-list form of kgat_peer_push: a pruned step exchanges only the rows of
 * "level 1 AND my range", not the whole slab. */
int kgat_peer_push_rows(const float* table, float* const* peer_tables, int32_t n_peers, const int32_t* rows,
                        const int32_t* count_dev, int64_t max_rows, int32_t d, int64_t ld, void* stream);
/* The same transfer on a copy engine (cudaMemcpyAsync into a peer mapping): no SM is involved, so it can run on a
 * side stream beside compute kernels without slowing them down.  One destination per call. */
int kgat_peer_copy(void* dst, const void* src, int64_t bytes, void* stream);
/* Channel handshake: seq[0] += 1; store it to *peer_flags[q] (my slot in peer q's flag pad) and wait until
 * my_flags[q] (written by peer q) has reached it, for every q < n_peers.  After it returns, everything the peers
 * stored into this rank's memory before *their* matching call is visible.  A wait longer than timeout_cycles SM
 * clocks sets status[0] = 1 and gives up (no hang).  peer_flags: DEVICE array of device pointers. */
int kgat_peer_signal_wait(int32_t* const* peer_flags, const int32_t* my_flags, int32_t n_peers, int32_t* seq, int32_t* status,
                          int64_t timeout_cycles, void* stream);

/* utility: fill used by the host glue so no torch kernel sits on the hot path */
int kgat_fill_f32(float* p, int64_t n, float value, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* host-latency helpers of the API fast path (the reference driver's per-step loop,               */
/* main.py:297-345: model(...), loss.backward(), update_*_weights(), loss.item())                */
/* ------------------------------------------------------------------------------------------- */
/* ring_host_mapped[s % n_slots] = (s << 32) | bits(*loss) with s = ++(*serial_dev): one aligned 8-byte store into
 * mapped pinned HOST memory (device-visible pointer), so the host can read a step's loss by polling without
 * synchronising the stream behind it. */
int kgat_publish_loss(const float* loss, uint64_t* serial_dev, uint64_t* ring_host_mapped, int32_t n_slots, void* stream);
/* cudaGraphLaunch(graph_exec, stream); graph_exec is a cudaGraphExec_t (host handle) */
int kgat_graph_launch(void* graph_exec, void* stream);
/* cudaMemcpyAsync(dst_dev, src, n_bytes, default kind, stream) followed by cudaGraphLaunch(graph_exec, stream):
 * the ids of one training step and the step itself in one call.  src: pinned host or device memory. */
int kgat_step_submit(void* dst_dev, const void* src, int64_t n_bytes, void* graph_exec, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KGAT_B200_H_ */
