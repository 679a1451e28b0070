/* hassaku_b200.h — C-ABI of the B200-native SGD matrix-factorization hot path.
 *
 * Drop-in boundary for ONE path of karapostK/hassaku (all citations are paths in that repository):
 *   train step   algorithms/base_classes.py:99-108, algorithms/sgd_alg.py:148-179, train/rec_losses.py:39-139,
 *                train/trainer.py:128-148 (+ torch.optim.AdamW, trainer.py:52-53), data/dataloader.py:56-57,92-129
 *   evaluator    eval/eval.py:54-99,101-118,237-253, eval/metrics.py:4-105
 * The reference has no FFI layer of its own (it is pure Python over torch); these are the entry points a
 * ctypes / torch-extension binding on the reference side calls — INTEGRATION.md shows that binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless stated otherwise; nothing here allocates
 *     device memory and nothing synchronises: all work is enqueued on `stream` (a cudaStream_t / CUstream)
 *   - every function returns HSK_OK (0) or a negative HSK_ERR_*; hsk_last_error() returns a thread-local text
 *   - embedding tables are fp32 row-major with a leading dimension `ld` (elements): ld % 4 == 0, ld >= d,
 *     base pointers 16-byte aligned, pad columns [d, ld) hold zeros (they stay zero under every kernel here);
 *     d <= 1024
 *   - indices are int64 like the reference loaders emit (data/dataloader.py:126-129)
 *   - `status` (nullable) is a device int32 bit-field: bit 0 is set when a kernel met an out-of-range user or
 *     item index (the offending sample is skipped; the reference would raise from torch at that point), bit 1 when a
 *     fixed-capacity exchange buffer of the item-sharded step overflowed (hsk_route_items), bit 2 when
 *     hsk_sample_negatives gave up on a row after its round cap (flagged slots were emitted)
 *   - the library is re-entrant and holds no mutable global state (nn.DataParallel calls forward from one
 *     Python thread per GPU, train/trainer.py:38-40); the current device of the calling thread is used
 */
#ifndef HASSAKU_B200_H
#define HASSAKU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* hsk_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define HSK_API __attribute__((visibility("default")))
#else
#define HSK_API
#endif

enum { HSK_OK = 0, HSK_ERR_INVALID = -1, HSK_ERR_CUDA = -2, HSK_ERR_UNSUPPORTED = -3 };
enum { HSK_LOSS_BPR = 0, HSK_LOSS_SAMPLED_SOFTMAX = 1, HSK_LOSS_BCE = 2 }; /* train/rec_losses.py:142-145 */
enum { HSK_STATUS_BAD_INDEX = 1, HSK_STATUS_CAPACITY = 2, HSK_STATUS_SAMPLER_ROUNDS = 4, HSK_STATUS_BARRIER_TIMEOUT = 8 };
enum { HSK_PREC_FP32 = 0, HSK_PREC_TF32 = 1, HSK_PREC_BF16 = 2 }; /* evaluator scoring precision */
/* kernel selection of hsk_mf_train_fused_v: every variant computes the same step (parity tests, A/B measurements) */
enum { HSK_TRAIN_AUTO = 0, HSK_TRAIN_REGS = 1, HSK_TRAIN_RING = 2, HSK_TRAIN_QWARP = 3 };
/* kernel selection of hsk_eval_topk_tc_v: one CTA per 128-user tile (cta_group::1) or CTA pairs (cta_group::2, the default) */
enum { HSK_EVAL_TC_AUTO = 0, HSK_EVAL_TC_SINGLE = 1, HSK_EVAL_TC_PAIR = 2 };

/* The embedding tables of one SGDMatrixFactorization (algorithms/sgd_alg.py:127-138).  Nullable: Ub, Ib, Gb. */
typedef struct hsk_mf_tables {
    float* Uw;        /* user_embeddings.weight  [n_users, ld]   */
    float* Vw;        /* item_embeddings.weight  [n_items, ld]   */
    float* Ub;        /* user_bias.weight        [n_users]  or NULL */
    float* Ib;        /* item_bias.weight        [n_items]  or NULL */
    float* Gb;        /* global_bias             [1]        or NULL */
    int64_t n_users;
    int64_t n_items;
    int32_t d;        /* embedding_dim */
    int32_t ld;       /* leading dimension of Uw and Vw (elements) */
} hsk_mf_tables;

HSK_API const char* hsk_last_error(void);
HSK_API int hsk_version(void);
/* sm count, compute capability, L2 bytes of the current device (host pointers, nullable) */
HSK_API int hsk_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* l2_bytes, int64_t* hbm_bytes);

/* ---- a1-a4: SGDBasedRecommenderAlgorithm.forward (base_classes.py:99-108; sgd_alg.py:148-179) -------------
 * scores[b, j] = <Uw[u_idx[b]], Vw[i_idx[b, j]]> (+ Ub[u]) (+ Ib[i]) (+ Gb), fp32, biases added after the
 * reduction like sgd_alg.py:171-178.  i_idx is [B, N1] row-major (column 0 = the positive). */
HSK_API int hsk_mf_scores(const hsk_mf_tables* t, const int64_t* u_idx, const int64_t* i_idx, int B, int N1,
                  float* scores /* [B, N1] */, int32_t* status, hsk_stream_t stream);

/* ---- a5-a6 (+bce): RecommenderSystemLoss.compute_loss (rec_losses.py:39-53, 68-88, 117-139) ---------------
 * Adds the batch-mean loss to *loss_accum (fp64, like the reference's float64 BPR loss) and, if dscores != NULL,
 * writes dL/dscores * grad_scale.  `labels` (nullable, fp64 [B, N1] like data/dataloader.py:127) defaults to
 * column 0 = 1, rest 0.  neg_shift = ln(n_items / neg_train) for sampled-softmax with uniform negatives
 * (rec_losses.py:133-134), else 0; if shifted_out != NULL the shifted logits are written there (it may alias
 * `scores`: the reference mutates the model output in place). */
HSK_API int hsk_rec_loss(const float* scores, const double* labels, int B, int N1, int loss_kind, float neg_shift,
                 float grad_scale, double* loss_accum, float* dscores /* [B, N1] or NULL */,
                 float* shifted_out /* [B, N1] or NULL */, hsk_stream_t stream);

/* ---- a7: backward of a1-a4 (autograd + aten::embedding_dense_backward in the reference) ------------------
 * Scatter-adds row gradients into DENSE gradient tables `g` (same layout as `t`, pre-zeroed by the caller or
 * left zero by hsk_adamw_dense):  gU[u_b] += sum_j ds_bj V[i_bj];  gV[i_bj] += ds_bj U[u_b];  gIb[i_bj] += ds_bj;
 * gUb[u_b] += sum_j ds_bj;  gGb += sum ds.  128-bit vector reductions (red.global.add.v4.f32). */
HSK_API int hsk_mf_scatter_grads(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                         const float* dscores, int B, int N1, int32_t* status, hsk_stream_t stream);

/* ---- a1-a7 in one pass: forward + loss + backward for one batch (train/trainer.py:133-146) ----------------
 * Each gathered row is read once: the dot product, the loss term, dL/ds and both row-gradient contributions
 * are produced while the row is in registers.  Adds the batch-mean loss to *loss_accum; accumulates into the
 * dense gradient tables `g`; optionally writes scores / dscores ([B, N1], nullable). */
HSK_API int hsk_mf_train_fused(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                       int B, int N1, int loss_kind, float neg_shift, double* loss_accum,
                       float* scores_out, float* dscores_out, int32_t* status, hsk_stream_t stream);

/* Item-sharded variant (SURVEY §8e): this rank holds B of the B_global samples of the step; the loss / gradient
 * normalisers stay GLOBAL (1 / (B_global N) for bpr, 1 / B_global for sampled-softmax, 1 / (B_global N1) for bce) so the
 * sum over ranks equals the single-GPU step on the whole batch.  `t->Vw` is then a compact table of fetched item rows. */
HSK_API int hsk_mf_train_fused_n(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                 int B, int N1, int64_t B_global, int loss_kind, float neg_shift, double* loss_accum,
                                 float* scores_out, float* dscores_out, int32_t* status, hsk_stream_t stream);

/* The same step with an explicit kernel choice: HSK_TRAIN_AUTO (what the two entry points above use: by shape, from the
 * B200 measurements), HSK_TRAIN_REGS (warp-per-row register gather), HSK_TRAIN_RING (bulk-copy / TMA row ring, bpr and
 * bce), HSK_TRAIN_QWARP (quarter-warp per sample, rows <= 128 floats).  A variant that does not support the shape falls
 * back to AUTO's choice.  Results agree within fp32 summation order. */
HSK_API int hsk_mf_train_fused_v(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                 int B, int N1, int64_t B_global, int loss_kind, float neg_shift, double* loss_accum,
                                 float* scores_out, float* dscores_out, int32_t* status, int variant, hsk_stream_t stream);

/* Row gather / scatter-add for the all-to-all exchanges of the item-sharded step: dst[r, :] = src[idx[r], :] and
 * dst[idx[r], :] += src[r, :] (128-bit vector reductions), rows of ld fp32 (ld % 4 == 0, 16-byte aligned). */
HSK_API int hsk_gather_rows(const float* src, int ld, const int64_t* idx, int64_t n, int64_t n_src, float* dst,
                            int32_t* status, hsk_stream_t stream);
HSK_API int hsk_scatter_add_rows(float* dst, int ld, const int64_t* idx, int64_t n, int64_t n_dst, const float* src,
                                 int32_t* status, hsk_stream_t stream);

/* ---- device-side routing of the item-sharded step's SPARSE exchange (SURVEY 8e): fixed shapes, no host sync, so the
 * whole step — these kernels, the NCCL all-to-alls between them, hsk_mf_train_fused_n, hsk_adamw_dense_rows — is one
 * CUDA graph.  World G: item i lives on rank i % G as local row i / G.
 *   hsk_route_items   (requester) the DISTINCT item ids among i_idx [n] (global ids), grouped by owner and numbered in
 *       ascending local-row order: req_rows [G, capq] int32 local rows wanted from each owner (-1 padded), req_count [G]
 *       (clamped to capq; an overflow sets HSK_STATUS_CAPACITY and the overflowing ids get compact index -1, which the
 *       train kernel reports as a bad index), compact_idx [n] int64 = q * block_rows + slot: the row of every batch slot in
 *       the compact table [G * block_rows, ld] of fetched rows, block_rows = hsk_shard_block_rows(capq, ld).
 *       No sort: presence flags over the owner-major id space + a 3-kernel exclusive scan (deterministic numbering).
 *   hsk_shard_pack    (owner) rows [G, capq] (what the peers sent after the id all-to-all) -> out [G, block_rows, ld]:
 *       block q = the requested rows of V, then from row capq on their item biases flat (Ib nullable).
 *   hsk_shard_unpack_add (owner) in [G, block_rows, ld] = the peers' row / bias gradients in the same layout:
 *       gV[row] += ..., gIb[row] += ..., stamps[row] = hsk_row_stamp(step) (nullable; for hsk_adamw_dense_rows).
 *   hsk_shard_unpack_ordered (owner) the same arguments; every row's gradient is composed in a fixed order and STORED
 *       (no floating-point atomics): see the order contract of the sharded 'ordered' step below.  It relies on what
 *       hsk_route_items guarantees of every request list rows[q, :]: the local rows are strictly ascending, followed by
 *       -1 padding only.
 *
 * ORDER CONTRACT of the sharded 'ordered' step (restated by tests/sharded_det_oracle.py: sharded_scatter_grads).  World G, item
 * i on rank i % G as local row i / G, user u on rank u % G; rank r processes the samples of the global batch whose user it
 * owns, in global batch order.
 *   1. Per rank: the single-GPU order contract (deterministic mode, below) on the local batch, with users keyed by local
 *      row and items keyed by their row in the compact table of fetched rows — owner-major, ascending local row within an
 *      owner, i.e. ordered exactly as (i % G) * cap + i / G.  Normalisers are global (B_global, hsk_mf_train_fused_det_n).
 *      The rank's user-row and user-bias gradients are final and stored.
 *   2. At the owner (hsk_shard_unpack_ordered): an item row's gradient, and its bias gradient, is the contributions of
 *      the ranks that fetched the row in increasing rank order: the first is stored, each later one added with fadd_rn.
 *      Rows no rank fetched are neither written nor stamped; stamps as hsk_shard_unpack_add.
 *   3. Global bias: every rank's chunked sum over its local slots (the contract below) is all-gathered and the G values
 *      are summed in rank order, starting from rank 0's value.
 *   4. Loss: every rank adds its fixed-order sum to its loss accumulator; the G fp64 accumulators are summed in rank order.
 *   At G = 1 this is the single-GPU deterministic step: the compact numbering is monotone in the item id. */
HSK_API int64_t hsk_shard_block_rows(int capq, int ld);
HSK_API int64_t hsk_route_scratch_bytes(int64_t n_items, int G);
HSK_API int hsk_route_items(const int64_t* i_idx, int64_t n, int64_t n_items, int G, int capq, int ld, int32_t* req_rows,
                            int32_t* req_count, int64_t* compact_idx, void* scratch, int64_t scratch_bytes,
                            int32_t* status, hsk_stream_t stream);
HSK_API int hsk_shard_pack(const float* V, const float* Ib /* nullable */, int ld, int64_t n_local, const int32_t* rows, int G,
                           int capq, float* out, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_shard_unpack_add(const float* in, int ld, int64_t n_local, const int32_t* rows, int G, int capq, float* gV,
                                 float* gIb /* nullable */, uint8_t* stamps /* nullable */, int64_t step,
                                 const int64_t* step_dev /* nullable: overrides step */, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_shard_unpack_ordered(const float* in, int ld, int64_t n_local, const int32_t* rows, int G, int capq, float* gV,
                                     float* gIb /* nullable */, uint8_t* stamps /* nullable */, int64_t step,
                                     const int64_t* step_dev /* nullable: overrides step */, int32_t* status,
                                     hsk_stream_t stream);

/* ---- evaluation over item SHARDS that stay where they are (one NVLink / NVSwitch node): every rank evaluates ITS users
 * against ALL items, streaming the other ranks' packed item tables straight from their HBM (TMA loads over peer mappings,
 * hsk_peer_export / hsk_peer_open) — no replica, no per-shard top-k, no merge.  Shard q (rank q) holds the items
 * q + n_shards * row.
 *   hsk_eval_topk_tc_shards   = hsk_eval_topk_tc over the shards' packed tables Vq_shards[q] [shard_rows[q], kpad] (from
 *       hsk_pack_rows) and item-bias vectors Ib_shards[q] (array or its entries nullable); CTA-pair kernel; ids returned
 *       are global; scratch >= hsk_eval_topk_tc_shards_scratch_bytes.
 *   hsk_rescore_topk_shards   = hsk_rescore_topk with the fp32 item rows read from the shards' tables V_shards[q]
 *       [shard_rows[q], t->ld]; t supplies the user side (Uw, Ub, Gb, n_users, d, ld). */
HSK_API int64_t hsk_eval_topk_tc_shards_scratch_bytes(int Be, const int64_t* shard_rows, int n_shards, int k);
HSK_API int hsk_eval_topk_tc_shards(const void* Uq, const void* const* Vq_shards, const int64_t* shard_rows,
                                    const float* const* Ib_shards, int n_shards, int kpad, int precision, const float* Ub,
                                    const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be, int64_t n_users,
                                    const int64_t* excl_indptr, const int32_t* excl_indices, int k, float* top_scores,
                                    int32_t* top_ids, void* scratch, int64_t scratch_bytes, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_rescore_topk_shards(const hsk_mf_tables* t, const float* const* V_shards, const int64_t* shard_rows,
                                    const float* const* Ib_shards, int n_shards, const int64_t* u_rows, int Be,
                                    const int32_t* cand_ids, const float* cand_scores /* nullable */, int n_cand, int k,
                                    float* top_scores, int32_t* top_ids, int32_t* status, hsk_stream_t stream);

/* ---- f3: FullEvaluatorCalibrationDecorator's recommendation distributions (eval/eval.py:174-179) ------------------
 * out[b, t, :] = (1 / ks[t]) * sum over j < ks[t] of item_tag[top_ids[b, j], :]   (top_ids int32 [B, k_list] ranked, -1 =
 * padding, skipped; item_tag fp32 [n_items, T] row-major; ks host array of n_ks <= 8 values, each <= k_list; out fp32
 * [B, n_ks, T]).  One pass over the ranked list per user instead of the reference's [B, k, T] gather. */
HSK_API int hsk_topk_tag_means(const int32_t* top_ids, int B, int k_list, const float* item_tag, int64_t n_items, int T,
                               const int* ks /* host */, int n_ks, float* out, int32_t* status, hsk_stream_t stream);

/* ---- PEER exchange of the item-sharded step: one kernel over NVLink peer memory instead of route / pack / all-to-all /
 * unpack (SURVEY 8e's exchange, fused into the step kernel).  Every rank of a node maps the item side of every other
 * rank's tables into its address space (CUDA IPC), then hsk_mf_train_fused_peer gathers the item rows of ITS samples
 * straight from their owners' HBM (128-byte loads over NVLink), and sends the row / bias gradients home as
 * red.relaxed.sys.global.add (performed in the owner's L2) together with the owner's row stamps
 * (hsk_adamw_dense_rows).  The caller brackets it with two cross-rank barriers per step: all peers' AdamW done -> kernel ->
 * all peers' kernels done -> AdamW.
 *   hsk_peer_export  handle of the device allocation that contains `ptr` + the offset of ptr in it (send both to the peers)
 *   hsk_peer_open    maps a peer's allocation: *base_out (keep for hsk_peer_close), the peer's `ptr` = base + offset;
 *                    open each distinct handle once per process
 *   hsk_mf_train_fused_peer  t / g: the LOCAL tables (user side used: Uw, Ub, Gb and their gradients; t->n_users local,
 *       t->n_items = the GLOBAL item count); peers->V[q] etc. = rank q's local item tables (own rank included), item i =
 *       row i / world of rank i % world; u_idx local rows, i_idx GLOBAL ids; normalisers from B_global as in
 *       hsk_mf_train_fused_n; stamps as hsk_shard_unpack_add.  Rows of at most 128 floats (quarter-warp kernel). */
#define HSK_MAX_PEERS 8
typedef struct hsk_peer_items {
    int32_t world;
    const float* V[HSK_MAX_PEERS];   /* [n_local_q, ld] */
    float* gV[HSK_MAX_PEERS];
    const float* Ib[HSK_MAX_PEERS];  /* all NULL or all set */
    float* gIb[HSK_MAX_PEERS];
    uint8_t* stamps[HSK_MAX_PEERS];  /* all NULL or all set */
} hsk_peer_items;
#define HSK_PEER_HANDLE_BYTES 64
HSK_API int hsk_peer_export(const void* ptr, void* handle /* [HSK_PEER_HANDLE_BYTES] */, int64_t* offset);
HSK_API int hsk_peer_open(const void* handle, void** base_out);
HSK_API int hsk_peer_close(void* base);
/* Cross-rank barrier on the stream (graph-capturable, no host argument changes between replays): every rank owns an
 * array of HSK_MAX_PEERS uint32 flags (zero-initialised, peer-mapped like the tables) and a local uint32 epoch counter
 * (zero-initialised).  The kernel bumps the epoch, stores it (st.release.sys) into flags[rank] of EVERY rank and spins
 * (ld.acquire.sys on its own flags) until every rank's epoch has arrived: work enqueued before the barrier on any rank
 * is complete before work enqueued after it starts on any rank.  All ranks must call it the same number of times; a
 * rank that waits longer than ~20 s gives up and sets HSK_STATUS_BARRIER_TIMEOUT. */
typedef struct hsk_peer_flags {
    int32_t world, rank;
    uint32_t* flags[HSK_MAX_PEERS];
} hsk_peer_flags;
HSK_API int hsk_peer_barrier(const hsk_peer_flags* f, uint32_t* epoch, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_mf_train_fused_peer(const hsk_mf_tables* t, const hsk_mf_tables* g, const hsk_peer_items* peers,
                                    const int64_t* u_idx, const int64_t* i_idx, int B, int N1, int64_t B_global, int loss_kind,
                                    float neg_shift, double* loss_accum, int64_t step,
                                    const int64_t* step_dev /* nullable: overrides step */, int32_t* status,
                                    hsk_stream_t stream);

/* Owner-sharded index arithmetic of the multi-GPU step (row i lives on rank i % world at local row i / world):
 * out[e] = (idx[e] % world) * rank_stride + idx[e] / world.  rank_stride = rows per rank of a rank-major replica
 * (dense exchange), or 0 for the plain local row.  Negative indices pass through unchanged so that the consumer's
 * bounds check still reports them.  out may alias idx. */
HSK_API int hsk_shard_local_index(const int64_t* idx, int64_t n, int world, int64_t rank_stride, int64_t* out,
                                  hsk_stream_t stream);

/* ---- a8: torch.optim.AdamW(params, lr, weight_decay).step over a flat fp32 range (trainer.py:52-53,147) ---
 * Dense decoupled-decay Adam over ALL n elements, every step (zero-gradient rows included), in one streaming
 * pass: reads p, m, v, g; writes p, m, v and (zero_grad != 0) g = 0, replacing optimizer.zero_grad().
 * `step` is the 1-based step count.  arith = 0 reproduces torch's CUDA foreach kernels bit for bit
 * (_multi_tensor_adam), arith = 1 torch's CPU single-tensor loop (_single_tensor_adam).  adam_l2 != 0 gives
 * torch.optim.Adam semantics (L2 added to the gradient instead of decoupled decay, trainer.py:48-49).
 * p, m, v, g 16-byte aligned. */
HSK_API int hsk_adamw_dense(float* p, float* m, float* v, float* g, int64_t n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int64_t step, int arith, int adam_l2, int zero_grad,
                    hsk_stream_t stream);

/* ---- the same dense update, skipping the gradient traffic of rows that received no gradient this step ---------------
 * Identical results to hsk_adamw_dense (bit for bit: an untouched row's gradient IS zero), but for the rows of the given
 * segments whose stamp byte differs from this step's stamp g is neither read nor re-zeroed: 24 B / element instead of
 * 32 B.  Contract: g is all-zero outside the rows stamped this step — hsk_adamw_dense_rows leaves it so, and every
 * caller that scatters gradients into rows calls hsk_mark_rows on their indices with the same step.  Everything
 * outside the segments (bias vectors, padding) takes the plain dense path, in the same launch: one kernel per call.
 * The stamp of step t is hsk_row_stamp(t) =
 * 1 + t % 255: the stamp arrays are never cleared (start them at 0).
 * Graph mode (both non-null): consts_dev = the 8 fp32 of hsk_adamw_consts for the step, step_dev = the 1-based step
 * count in device memory (it selects the stamp), so that one captured launch serves every step; lr ... step are then
 * ignored.  Only decoupled AdamW / Adam(L2) / plain Adam like hsk_adamw_dense; the gradient is always zeroed. */
typedef struct hsk_row_segment {
    int64_t offset;          /* first element of the segment inside p / m / v / g (multiple of 4) */
    int64_t n_rows;
    int32_t ld;              /* elements per row (multiple of 4) */
    const uint8_t* stamps;   /* [n_rows] device bytes */
} hsk_row_segment;
HSK_API int hsk_row_stamp(int64_t step);
HSK_API int hsk_mark_rows(const int64_t* idx, int64_t n, int64_t n_rows, uint8_t* stamps, int64_t step,
                          const int64_t* step_dev /* nullable: overrides step */, hsk_stream_t stream);
/* both tables of one training batch in one launch: stamps_users[u_idx[b]] = stamps_items[i_idx[b, j]] = stamp (nullable each) */
HSK_API int hsk_mark_batch(const int64_t* u_idx, const int64_t* i_idx, int B, int N1, int64_t n_users, int64_t n_items,
                           uint8_t* stamps_users, uint8_t* stamps_items, int64_t step, const int64_t* step_dev,
                           hsk_stream_t stream);
HSK_API int hsk_adamw_dense_rows(float* p, float* m, float* v, float* g, int64_t n, const hsk_row_segment* segments /* host */,
                                 int n_segments /* <= 4 */, double lr, double beta1, double beta2, double eps,
                                 double weight_decay, int64_t step, const float* consts_dev, const int64_t* step_dev,
                                 int arith, int adam_l2, hsk_stream_t stream);

/* ---- hsk_adamw_dense_rows with the moments of untouched rows written back once every `lag` steps ---------------------
 * p after every call, and m and v after hsk_adamw_lag_sync, are bit for bit those of hsk_adamw_dense_rows with the same
 * arguments.  A row of a segment keeps the m and v of the step `base` at which they were last written; a call replays
 * the steps without gradient since then in registers (m and v of such a step depend on beta1, beta2 and the old values
 * only), applies step `step`, stores p, and writes m and v back (base = step) only when the row is stamped this step or
 * (step + row) % lag == 0 — else 16 instead of 24 bytes per parameter.  Everything outside the segments is updated as in
 * hsk_adamw_dense_rows.  lag = 1 writes every row every step: hsk_adamw_dense_rows exactly.
 * base_in[s] / base_out[s] (host arrays of n_segments device pointers; for every non-empty segment two distinct
 * [n_rows] byte arrays): base & 255 per row is read from base_in and written to base_out for every row; the caller
 * swaps them after the call.  Contract: 1 <= step - base <= lag for every row — start a segment with base = step - 1 of
 * its first call (its m and v current), call with consecutive steps, and sync before any other update of m and v, a
 * change of beta1 / beta2 / arith / lag, or a read of m and v.  Only AdamW (decoupled decay) or Adam with
 * weight_decay = 0: L2 decay gives untouched rows a non-zero gradient.  No graph mode (consts_dev / step_dev). */
HSK_API int hsk_adamw_dense_rows_lag(float* p, float* m, float* v, float* g, int64_t n,
                                     const hsk_row_segment* segments /* host */, int n_segments /* <= 4 */,
                                     const uint8_t* const* base_in /* host */, uint8_t* const* base_out /* host */,
                                     int lag /* 1..128 */, double lr, double beta1, double beta2, double eps,
                                     double weight_decay, int64_t step, int arith, int adam_l2, hsk_stream_t stream);
/* every row of the segments to step `step` (the last step taken): replays its steps without gradient since base_in,
 * writes m and v, and sets base_out = step for every row (swap after the call).  The segments' stamps are not read. */
HSK_API int hsk_adamw_lag_sync(float* m, float* v, int64_t n, const hsk_row_segment* segments /* host */,
                               int n_segments /* <= 4 */, const uint8_t* const* base_in /* host */,
                               uint8_t* const* base_out /* host */, double beta1, double beta2, int64_t step, int arith,
                               hsk_stream_t stream);

/* ---- a10: uniform negative sampling on the device (data/dataloader.py:56-57, 92-129) -------------------------------
 * For every batch row b: i_idx[b, 0] = pos_idx[b] (if pos_idx != NULL) and i_idx[b, 1..N] = N items drawn uniformly
 * from [0, n_items) none of which is a TRAIN item of user u_idx[b] (CSR of the training interactions: indptr int64
 * [n_users + 1], indices int32 sorted per row), redrawing flagged slots until the row is clean — the reference's
 * collate loop.  distinct_in_row != 0 additionally redraws a slot when a higher slot of the row holds the same item
 * (numpy's assume_unique sort path; the reference's common case).  Stream: Philox4x32-10 keyed by (seed, step), a
 * pure function of (seed, step, b, slot) — restated bit-exactly by oracle/philox.py.  i_idx is [B, 1 + N] int64.
 * pop_cdf (nullable): 'popular' strategy (data/dataloader.py:59-64, item ~ pop^alpha): a 64-bit fixed-point CDF over the
 * items, cdf[i] = floor(2^64 * sum_{t<=i} p_t) with cdf[n_items-1] = 2^64 - 1; NULL = uniform. */
HSK_API int hsk_sample_negatives(const int64_t* u_idx, const int64_t* pos_idx /* nullable */, int B, int N, int64_t n_items,
                                 int64_t n_users, const int64_t* csr_indptr, const int32_t* csr_indices, uint64_t seed,
                                 uint64_t step, int distinct_in_row, const uint64_t* pop_cdf /* nullable */, int64_t* i_idx,
                                 int32_t* status, hsk_stream_t stream);

/* ==== full-rank evaluator (eval/eval.py:54-99, 101-118, 237-253; eval/metrics.py:4-105) ========================= */

/* ---- a12 + top-k of a14: evaluate_recommender_algorithm's SGD branch for one user batch (eval.py:243-253, :63) ---
 * For every user u_idx[r], r < Be: scores against ALL rows of the item table `t->Vw` (this GPU's item shard;
 * local row j has global item id id_offset + j * id_stride), score = <U_u, V_j> (+ Ub) (+ Ib) (+ Gb) in fp32
 * (eval.py:247-248), -inf on every id in the user's exclusion row (CSR, sorted global ids, int32; eval.py:250-251),
 * then the k best: top_scores/top_ids [Be, k], ordered by score descending, ties by item id ascending (torch.topk
 * leaves tie order unspecified).  Slots beyond the number of items get id -1 / score -inf.  The [Be, I] score matrix
 * is never materialised.  `scratch`: hsk_eval_topk_scratch_bytes(Be, t->n_items, k) bytes of device memory.
 * u_rows (nullable): when the user rows were gathered from other GPUs (item-sharded evaluation) batch entry r reads row
 * u_rows[r] of t->Uw / t->Ub while u_idx[r] stays the GLOBAL user id (< n_users_global) that selects the exclusion row. */
HSK_API int64_t hsk_eval_topk_scratch_bytes(int Be, int64_t n_local_items, int k);
HSK_API int hsk_eval_topk(const hsk_mf_tables* t, const int64_t* u_idx, const int64_t* u_rows /* nullable */,
                          int64_t n_users_global, int Be, int64_t id_offset, int64_t id_stride,
                          const int64_t* excl_indptr /* [n_users + 1] or NULL */, const int32_t* excl_indices,
                          int k /* <= 128 */, float* top_scores, int32_t* top_ids, void* scratch, int64_t scratch_bytes,
                          int32_t* status, hsk_stream_t stream);

/* ---- the same on the tensor cores (TF32 / BF16 mode): tcgen05.mma with TMEM accumulators, TMA-fed, fused epilogue ------
 * Operands are packed copies of the tables: Uq = the user batch's rows [Be, kpad], Vq = the item shard [n_local, kpad],
 * row-major, bf16 (HSK_PREC_BF16) or tf32-rounded fp32 (HSK_PREC_TF32), zero padded to kpad = hsk_eval_tc_kpad(d, prec)
 * — build them with hsk_pack_rows (row_idx = u_idx gathers the batch; row_idx = NULL packs a whole table).
 * Biases stay fp32 and are added in the epilogue (Ub is the user-bias TABLE, indexed by u_idx).  Everything else as
 * hsk_eval_topk, including the tail: a user with fewer than k admissible items gets them first, then the ids of the
 * user's exclusion row at score -inf, lowest id first, then id -1 / score -inf once both run out.
 * Supports kpad * element size <= 1024 bytes (d <= 512 bf16, d <= 256 tf32). */
HSK_API int hsk_eval_tc_kpad(int d, int precision);
HSK_API int hsk_pack_rows(const float* src, int ld, int d, const int64_t* row_idx /* nullable */, int64_t n_out, int64_t n_src,
                          void* dst, int kpad, int precision, int32_t* status, hsk_stream_t stream);
HSK_API int64_t hsk_eval_topk_tc_scratch_bytes(int Be, int64_t n_local_items, int k);
HSK_API int hsk_eval_topk_tc(const void* Uq, const void* Vq, int kpad, int precision, const float* Ub, const float* Ib,
                             const float* Gb, const int64_t* u_idx, const int64_t* u_rows /* nullable: rows of Ub */, int Be,
                             int64_t n_users, int64_t n_local,
                             int64_t id_offset, int64_t id_stride, const int64_t* excl_indptr, const int32_t* excl_indices,
                             int k, float* top_scores, int32_t* top_ids, void* scratch, int64_t scratch_bytes,
                             int32_t* status, hsk_stream_t stream);

/* The same with an explicit kernel choice (parity tests, A/B measurements): HSK_EVAL_TC_PAIR = thread-block clusters of two
 * CTAs, tcgen05.mma.cta_group::2 with M = 256 / N = 256 tiles, the item tile shared by the pair, item bias pre-loaded into
 * the TMEM accumulator (default); HSK_EVAL_TC_SINGLE = one CTA per 128-user tile, M = N = 128.  Both return the same
 * ranking up to the rounding of (bias + dot) against (dot + bias). */
HSK_API int hsk_eval_topk_tc_v(const void* Uq, const void* Vq, int kpad, int precision, const float* Ub, const float* Ib,
                               const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be, int64_t n_users,
                               int64_t n_local, int64_t id_offset, int64_t id_stride, const int64_t* excl_indptr,
                               const int32_t* excl_indices, int k, float* top_scores, int32_t* top_ids, void* scratch,
                               int64_t scratch_bytes, int32_t* status, int variant, hsk_stream_t stream);

/* ---- fp32 re-scoring of tensor-core candidates: TF32 / BF16 ranking, fp32 scores and order ------------------------------
 * cand_ids [Be, n_cand] (n_cand <= 128; global item ids as hsk_eval_topk_tc returns them, < 0 = empty, exclusions already
 * removed): every candidate is scored again from the fp32 tables `t` (score = <Uw[u_rows[r]], Vw[(id - id_offset) /
 * id_stride]> (+ Ub[u_rows[r]]) (+ Ib) (+ Gb), eval/eval.py:247-248) and the k best are returned ordered like
 * hsk_eval_topk (score descending, lower id first).  Call hsk_eval_topk_tc with k' = n_cand = min(128, k + 28), then
 * this: the result differs from the fp32 evaluator only if a true top-k item fell below rank n_cand in the
 * low-precision pass.  u_rows [Be] = rows of t->Uw / t->Ub (< t->n_users).  cand_scores (nullable, [Be, n_cand]: the
 * low-precision scores): a candidate whose score is -inf is an item of the user's exclusion row that surfaced because
 * fewer than n_cand admissible items exist; it keeps -inf (and so sorts after every admissible item). */
HSK_API int hsk_rescore_topk(const hsk_mf_tables* t, const int64_t* u_rows, int Be, int64_t id_offset, int64_t id_stride,
                             const int32_t* cand_ids, const float* cand_scores /* nullable */, int n_cand, int k,
                             float* top_scores, int32_t* top_ids, int32_t* status, hsk_stream_t stream);

/* Item-sharded evaluation re-scores AFTER the merge, so that the fp32 work shards with the items (each shard scores only
 * the merged candidates it owns, ~n_cand / G per user) instead of every shard re-scoring its own n_cand:
 *   hsk_rescore_scores  positional: out_scores[r, c] = the fp32 score of cand_ids[r, c] if this shard owns it
 *                       ((id - id_offset) % id_stride == 0), else -inf (ids of other shards are expected here);
 *   hsk_topk_combine    on the row's owner: scores [G, rows, n_cand] from all shards + the merged ids [rows, n_cand] ->
 *                       candidate score = max over shards, then the k best ordered like hsk_eval_topk.  cand_scores
 *                       (nullable, [rows, n_cand]: the merged low-precision scores): -inf marks an excluded item of
 *                       the tail, which stays -inf as in hsk_rescore_topk. */
HSK_API int hsk_rescore_scores(const hsk_mf_tables* t, const int64_t* u_rows, int Be, int64_t id_offset, int64_t id_stride,
                               const int32_t* cand_ids, int n_cand, float* out_scores /* [Be, n_cand] */, int32_t* status,
                               hsk_stream_t stream);
HSK_API int hsk_topk_combine(const float* scores, const int32_t* ids, const float* cand_scores /* nullable */, int G, int rows,
                             int n_cand, int k, float* out_scores, int32_t* out_ids, hsk_stream_t stream);

/* ---- merge of G per-shard top-k lists (item-sharded evaluation: all-gather, then this) --------------------------
 * scores/ids: [G, rows, k] (id < 0 = empty slot) -> out [rows, k], same ordering rule as hsk_eval_topk. */
HSK_API int hsk_topk_merge(const float* scores, const int32_t* ids, int G, int rows, int k, float* out_scores,
                           int32_t* out_ids, hsk_stream_t stream);

/* ---- logits.topk(k) of a dense [rows, n_cols] fp32 matrix: FullEvaluator.eval_batch's dense API (eval.py:61-63) -- */
HSK_API int hsk_topk_dense(const float* logits, int rows, int64_t n_cols, int64_t row_stride, int k, float* out_scores,
                           int32_t* out_ids, hsk_stream_t stream);

/* ---- a14-a17: precision / recall / ndcg @ ks (eval/metrics.py:4-105) and their per-group sums (eval.py:66-99) ----
 * top_ids [Be, k_max] ranked item ids (id < 0 = empty); labels as CSR rows of the evaluation split (sorted int32 item
 * ids per user) or, in the _dense variant, y_true [Be, n_items] fp32 0/1 rows (the reference's dense API).
 * discount [k_max] fp32 = 1 / log2(r + 2).  Per user and cut-off ks[t]: precision = hits / k; recall = hits / n+
 * (0 if the user has no positives); ndcg = min(1, dcg / idcg) (0 if no positives).  Adds into
 * sums [(1 + n_groups), n_ks, 3] (fp64; row 0 = all users, row 1 + g = users with user_group[u] == g) and
 * counts [1 + n_groups] (int64); if per_user != NULL also writes [Be, n_ks, 3] fp32.  The caller zeroes sums/counts
 * at the start of a sweep and reads them once at the end (one host sync per sweep instead of >= 12 per batch). */
HSK_API int hsk_rank_metrics(const int32_t* top_ids, int Be, int k_max, const int* ks /* host */, int n_ks,
                             const int64_t* u_idx, const int64_t* lab_indptr, const int32_t* lab_indices,
                             const int32_t* user_group /* [n_users] or NULL */, int n_groups, const float* discount,
                             float* per_user, double* sums, int64_t* counts, hsk_stream_t stream);
HSK_API int hsk_rank_metrics_dense(const int32_t* top_ids, int Be, int k_max, const int* ks /* host */, int n_ks,
                                   const int64_t* u_idx, const float* y_true, int64_t n_items,
                                   const int32_t* user_group, int n_groups, const float* discount, float* per_user,
                                   double* sums, int64_t* counts, hsk_stream_t stream);

/* ---- torch.optim.Adagrad(params, lr, weight_decay).step (train/trainer.py:50-51), dense, op order of torch's CUDA foreach
 * path (lr_decay 0, eps default 1e-10): g += wd p; sum += g g; p -= lr g / (sqrt(sum) + eps); g zeroed if zero_grad. */
HSK_API int hsk_adagrad_dense(float* p, float* state_sum, float* g, int64_t n, double lr, double eps, double weight_decay,
                              int zero_grad, hsk_stream_t stream);

/* ---- row-sparse "lazy" AdamW (reported separately: NOT torch.optim.AdamW's trajectory) ------------------------------
 * hsk_mark_touched sets touched_users[u] = touched_items[i] = 1 for every index of the batch; hsk_adamw_rows_lazy then
 * updates p, m, v (and zeroes g) ONLY for rows whose flag is set and clears the flag — torch.optim.SparseAdam semantics
 * (global step count for the bias corrections) plus decoupled weight decay on the touched rows.  `*_bias` (nullable)
 * are the length-n_rows vectors sharing the row index (item_bias with the item table, user_bias with the user table). */
HSK_API int hsk_mark_touched(const int64_t* u_idx, const int64_t* i_idx, int B, int N1, int64_t n_users, int64_t n_items,
                             uint8_t* touched_users, uint8_t* touched_items, hsk_stream_t stream);
HSK_API int hsk_adamw_rows_lazy(float* p, float* m, float* v, float* g, int64_t n_rows, int ld, float* p_bias, float* m_bias,
                                float* v_bias, float* g_bias, uint8_t* touched, double lr, double beta1, double beta2,
                                double eps, double weight_decay, int64_t step, hsk_stream_t stream);

/* ---- CUDA-graph friendly AdamW: the step-dependent scalars live in device memory --------------------------------------
 * hsk_adamw_consts fills 8 fp32 (HOST) for step `step`; the caller copies them to `consts_dev` (captured as a memcpy
 * node from pinned memory) and hsk_adamw_dense_graph applies exactly the arithmetic of hsk_adamw_dense(arith = 0) with
 * them, so one captured graph serves every step.  decoupled_decay / adam_l2 select AdamW / Adam(L2) / plain Adam. */
HSK_API int hsk_adamw_consts(double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                             float* out8 /* host */);
HSK_API int hsk_adamw_dense_graph(float* p, float* m, float* v, float* g, int64_t n, const float* consts_dev,
                                  int decoupled_decay, int adam_l2, int zero_grad, hsk_stream_t stream);

/* ==== trial pack: M models of one shape (a hyperparameter sweep) trained by one launch per kernel ====================
 * The M parameter arenas are the rows of one [M, trial_stride] fp32 allocation (m, v and the gradient arena likewise):
 * trial j's tables are trial 0's tables + j * trial_stride elements.  trial_stride % 4 == 0, so with trial 0's tables
 * 16-byte aligned every trial's are.  `active` (device int32 [n_active]) lists the trials a launch works on; one grid
 * dimension walks it, so an inactive trial costs no CTA and none of its memory is read or written.  An entry outside
 * [0, n_trials) sets HSK_STATUS_BAD_INDEX in `status` and that entry's work is skipped.  n_active <= 65535.
 *   hsk_mf_train_fused_pack  hsk_mf_train_fused for every active trial on ONE shared batch u_idx / i_idx: t / g = trial
 *       0's parameter / gradient tables, loss_accum [n_trials] fp64 (trial j adds its batch-mean loss to loss_accum[j]).
 *       Kernel and item-slot split follow HSK_TRAIN_AUTO's rules applied to n_active * B samples, with the
 *       register-gather kernel wherever AUTO would take the bulk-copy ring.  Scores / dscores are not written.
 *   hsk_adamw_pack  hsk_adamw_dense (arith 0, gradient zeroed) for every active trial, in one streaming pass:
 *       consts_dev [n_trials, 8] fp32 = each trial's hsk_adamw_consts for this step (16-byte aligned).  adam_l2 = 0:
 *       AdamW; 1: Adam(L2).  A trial whose wd entry is 0 gets no weight-decay term, as torch does for wd == 0 (torch tests
 *       the double: the two agree unless 0 < |wd| < 2^-150).  n_segments > 0 is the row-stamped form of
 *       hsk_adamw_dense_rows: `segments` are offsets inside ONE trial's row (0 <= offset, end <= trial_stride), the stamp
 *       arrays are shared by every trial (every trial saw the same batch) and `step` (>= 1) selects the stamp; outside
 *       the segments the row takes the dense path in the same launch.  Bitwise identical to hsk_adamw_dense /
 *       hsk_adamw_dense_rows with arith 0 per trial.
 *   hsk_adamw_consts_table  host: out [n_steps, n_trials, 8] = hsk_adamw_consts(lr[j], ..., weight_decay[j], first_step +
 *       s) for every step s and trial j (one table per epoch: no per-step host work or copy). */
HSK_API int hsk_mf_train_fused_pack(const hsk_mf_tables* t, const hsk_mf_tables* g, int64_t trial_stride, int n_trials,
                                    const int32_t* active, int n_active, const int64_t* u_idx, const int64_t* i_idx, int B,
                                    int N1, int loss_kind, float neg_shift, double* loss_accum /* [n_trials] */,
                                    int32_t* status, hsk_stream_t stream);
HSK_API int hsk_adamw_pack(float* p, float* m, float* v, float* g, int64_t trial_stride, int n_trials, const int32_t* active,
                           int n_active, const float* consts_dev, const hsk_row_segment* segments /* host, nullable */,
                           int n_segments /* <= 4 */, int64_t step, int adam_l2, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_adamw_consts_table(const double* lr /* host [n_trials] */, const double* weight_decay /* host [n_trials] */,
                                   int n_trials, double beta1, double beta2, double eps, int64_t first_step, int n_steps,
                                   float* out /* host [n_steps, n_trials, 8] */);

/* ---- packed validation: the fp32 evaluator and its metrics for every active trial of a pack in one launch each ---------
 * Same layout and `active` rules as above (an out-of-range entry sets HSK_STATUS_BAD_INDEX and its CTAs write nothing;
 * its output rows are then undefined).  Single GPU: no id mapping, u_rows or item shards.
 *   hsk_eval_topk_pack  hsk_eval_topk (fp32, id_offset 0, id_stride 1) of every active trial on ONE shared user batch
 *       u_idx [Be] and ONE shared exclusion CSR: top_scores / top_ids [n_active, Be, k], row a * Be + r = trial active[a],
 *       user u_idx[r].  Each row is bitwise what hsk_eval_topk returns for that trial and user, whatever Be and n_active
 *       (a row's per-item arithmetic and key order do not depend on the launch shape).  The item split plan counts
 *       n_active times the row tiles, so items are not split where the trials already fill the GPU; scratch:
 *       hsk_eval_topk_pack_scratch_bytes(Be, t->n_items, k, n_active) bytes.  n_active * Be < 2^31.
 *   hsk_rank_metrics_pack  hsk_rank_metrics (CSR labels) of top_ids [n_active, Be, k_max]: trial active[a] adds into its
 *       own slices sums [n_trials, 1 + n_groups, n_ks, 3] (fp64) and counts [n_trials, 1 + n_groups]; per_user (nullable)
 *       [n_active, Be, n_ks, 3].
 *   hsk_rank_metrics_sums_det_pack  hsk_rank_metrics_sums_det for per_user [n_active, Be, n_ks, 3] into the same sums
 *       layout: each trial's Be rows are cut into consecutive batches of `batch` rows (the last may be shorter) and
 *       added batch by batch, in order — bitwise what one hsk_rank_metrics_sums_det call per batch gives. */
HSK_API int64_t hsk_eval_topk_pack_scratch_bytes(int Be, int64_t n_items, int k, int n_active);
HSK_API int hsk_eval_topk_pack(const hsk_mf_tables* t, int64_t trial_stride, int n_trials, const int32_t* active, int n_active,
                               const int64_t* u_idx, int Be, const int64_t* excl_indptr /* [n_users + 1] or NULL */,
                               const int32_t* excl_indices, int k /* <= 128 */, float* top_scores, int32_t* top_ids,
                               void* scratch, int64_t scratch_bytes, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_rank_metrics_pack(const int32_t* top_ids, int Be, int k_max, const int* ks /* host */, int n_ks,
                                  const int64_t* u_idx, const int64_t* lab_indptr, const int32_t* lab_indices,
                                  const int32_t* user_group /* [n_users] or NULL */, int n_groups, const float* discount,
                                  int n_trials, const int32_t* active, int n_active, float* per_user /* nullable */,
                                  double* sums, int64_t* counts, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_rank_metrics_sums_det_pack(const float* per_user, int Be, int batch, int n_ks, const int64_t* u_idx,
                                           const int32_t* user_group /* nullable */, int n_groups, int n_trials,
                                           const int32_t* active, int n_active, double* sums, int32_t* status,
                                           hsk_stream_t stream);

/* ==== deterministic mode (hsk_det.cu): bitwise-reproducible training / evaluation reductions ========================
 * What the Python layer runs under torch.use_deterministic_algorithms(True).  The batch is grouped by row (stable radix
 * sort of the item ids of the B * N1 slots and of the user ids of the B samples) and every touched row is produced by ONE
 * warp as a fixed-order sum: no floating-point atomics, the same bits on every run, grid and GPU.
 * Order (restated bit for bit by oracle/det_oracle.py): slot s = b * N1 + j; a row's entries are taken in increasing s;
 * they are cut into chunks at the row's ends and at every multiple of C = 32 of the entry's position in the sorted list
 * (the user list expands every sample into its N1 slots); within a chunk acc = +0, acc = fadd_rn(acc, fmul_rn(ds_s,
 * other_row)) (other_row = Uw[u_b] for an item row, Vw[i_s] for a user row; bias: acc_b = fadd_rn(acc_b, ds_s)); the
 * row is the chunk partials added in order from the first.  gGb: chunks of 1024 consecutive slots, the same way.
 * Unlike hsk_mf_scatter_grads the rows are STORED: every row the batch touches is overwritten with its gradient (g must
 * be zero there to get the same result as the accumulating kernels); rows it does not touch are not written.
 * Scratch: device memory of hsk_det_scratch_bytes(B, N1, ld) bytes, 16-byte aligned, owned by the caller.
 *   hsk_mf_scatter_grads_det   = hsk_mf_scatter_grads with the order above.  An entry whose user / item is out of range is
 *       skipped and reported in status.
 *   hsk_mf_train_fused_det     = hsk_mf_train_fused: per sample the fused kernels' scores, loss term and dL/ds (a sample
 *       with an out-of-range index is skipped: dL/ds 0, loss 0), then the scatter above; *loss_accum += the per-sample
 *       fp64 losses summed in a fixed order.  N1 <= 10240.
 *   hsk_mf_train_fused_det_n   = hsk_mf_train_fused_det with the loss / gradient normalisers of a global batch of
 *       B_global >= B samples (as hsk_mf_train_fused_n): one rank's share of the sharded 'ordered' step.  B = 0 (a rank
 *       without samples) launches nothing and accepts null index pointers.
 *   hsk_rec_loss_det           = hsk_rec_loss (dscores required, not aliasing scores) with the per-row losses summed in a
 *       fixed order; scratch >= 8 * B bytes.
 *   hsk_rank_metrics_sums_det  sums[g] += the fixed-order sum of per_user [Be, n_ks, 3] (hsk_rank_metrics' per-user
 *       output) over the batch's users of group g - 1 (g = 0: all users), g < 1 + n_groups: the deterministic
 *       replacement of hsk_rank_metrics' floating-point sums (its integer counts are exact as they are). */
HSK_API int64_t hsk_det_scratch_bytes(int B, int N1, int ld);
HSK_API int hsk_mf_scatter_grads_det(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                     const float* dscores, int B, int N1, void* scratch, int64_t scratch_bytes, int32_t* status,
                                     hsk_stream_t stream);
HSK_API int hsk_mf_train_fused_det(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                   int B, int N1, int loss_kind, float neg_shift, double* loss_accum, float* scores_out,
                                   float* dscores_out, void* scratch, int64_t scratch_bytes, int32_t* status, hsk_stream_t stream);
HSK_API int hsk_mf_train_fused_det_n(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                     int B, int N1, int64_t B_global, int loss_kind, float neg_shift, double* loss_accum,
                                     float* scores_out, float* dscores_out, void* scratch, int64_t scratch_bytes,
                                     int32_t* status, hsk_stream_t stream);
HSK_API int hsk_rec_loss_det(const float* scores, const double* labels, int B, int N1, int loss_kind, float neg_shift,
                             float grad_scale, double* loss_accum, float* dscores, float* shifted_out /* nullable */,
                             void* scratch, int64_t scratch_bytes, hsk_stream_t stream);
HSK_API int hsk_rank_metrics_sums_det(const float* per_user, int Be, int n_ks, const int64_t* u_idx,
                                      const int32_t* user_group /* nullable */, int n_groups, double* sums, hsk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* HASSAKU_B200_H */
