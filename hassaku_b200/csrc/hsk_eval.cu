// a12-a17 — full-rank evaluator kernels (eval/eval.py:54-99, 237-253; eval/metrics.py:4-105), fp32-exact mode.
//
//   hsk_eval_topk     scores = U_b · V^T (+ biases) for a user batch against an item shard, -inf on the user's
//                     excluded (train / train+val) items, running top-k — fused: the [Be, I] score matrix is never
//                     written to memory (the reference materialises [Be, I, d], sgd_alg.py:171)
//   hsk_topk_merge    k-way merge of per-split / per-GPU top-k lists
//   hsk_topk_dense    top-k of a dense logits matrix (FullEvaluator.eval_batch's dense API, eval.py:61-63)
//   hsk_rank_metrics  precision / recall / ndcg @ ks from top-k ids + CSR labels, per-group sums on device
//   hsk_rank_metrics_dense   same from dense y_true rows (the reference's dense API)
//   hsk_eval_topk_pack / hsk_rank_metrics_pack   the same two for every active trial of a trial pack in one launch
//
// fp32-exact scoring is a classic SIMT FFMA tile kernel (64 users x 128 items per CTA, 16-wide K chunks staged by
// cp.async double buffering, 4x8 accumulators per thread): north_star requires bit-exact top-k ids against the fp32
// reference, which rules tensor-core input rounding out for this mode; the TF32/BF16 tcgen05 path is hsk_eval_tc.cu.
#include "hsk_topk.cuh"

namespace hsk {

constexpr int TM = 64;     // users per CTA
constexpr int TN = 128;    // items per tile
constexpr int KC = 16;     // K chunk
constexpr int KP = 20;     // padded smem row (floats): conflict-free 128-bit reads for the strided thread map
constexpr int kEvalThreads = 256;
constexpr int EV_KPL = 16;            // candidate keys per lane: 512-entry lists (a 256-entry list with k = 100 left only
constexpr int EV_CAP = 32 * EV_KPL;   // 28 entries of slack per 128-item tile and was re-sorted at almost every tile)

struct EvalArgs {
    const float* __restrict__ Uw;
    const float* __restrict__ Vw;   // item shard, local rows
    const float* __restrict__ Ub;
    const float* __restrict__ Ib;   // local rows
    const float* __restrict__ Gb;
    const int64_t* __restrict__ u_idx;
    const int64_t* __restrict__ u_rows;   // row of Uw / Ub per batch entry (null: = u_idx)
    int64_t n_urows;
    const int64_t* __restrict__ excl_indptr;
    const int32_t* __restrict__ excl_indices;
    int64_t n_users;
    int64_t n_local;         // items in this shard
    int64_t id_offset, id_stride;   // global item id of local row j = id_offset + j * id_stride
    int ld, Be, k;
    int n_tiles, tiles_per_split, n_splits;
    uint64_t* cand;          // [n_splits, Be, EV_CAP]
    float* out_scores;       // [Be, k]  (written directly when n_splits == 1)
    int32_t* out_ids;
    int32_t* status;
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
    const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void write_topk_row(const uint64_t* list, int k, float* out_s, int32_t* out_i, int lane) {
    for (int e = lane; e < k; e += 32) {
        const uint64_t key = list[e];
        out_s[e] = key ? key_score(key) : -INFINITY;
        out_i[e] = key_id(key);
    }
}

// out-of-line: the list cut (radix select + fallback sort network) is rare and large; inlined into the tile loop it also
// made the compiler's unroller explode
__device__ __noinline__ int ev_cut(uint64_t* list, int n, int n_checked, int k, int lane, const int32_t* __restrict__ excl,
                                   int64_t lo, int64_t hi, float* new_tau, uint64_t* new_taukey) {
    return warp_cut_list<EV_KPL>(list, n, n_checked, k, kCap - TN, lane, excl, lo, hi, new_tau, new_taukey);
}
__device__ __noinline__ void ev_final_sort(uint64_t* list, int n, int k, int lane) {
    uint64_t thr;
    warp_prune_list<kKeysPerLane>(list, n, k, lane, &thr);
}

__global__ void __launch_bounds__(kEvalThreads, 2) eval_topk_f32_kernel(EvalArgs a) {
#define EV_SPLIT_ROWS a.Be
#include "hsk_eval_topk_body.inc"
#undef EV_SPLIT_ROWS
}

// ---- merge of G sorted key lists per row (lists[g] at base + (g * rows + row) * stride) ----
__global__ void __launch_bounds__(256) topk_merge_keys_kernel(const uint64_t* __restrict__ lists, int G, int rows,
                                                              int stride, int k, float* out_s, int32_t* out_i,
                                                              const float* __restrict__ Ub, const float* __restrict__ Gb,
                                                              const int64_t* __restrict__ u_idx, int64_t n_users) {
    __shared__ uint64_t buf[8][kCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x * 8 + warp;
    if (row >= rows) return;
    uint64_t* mine = buf[warp];
    for (int e = lane; e < kCap; e += 32) mine[e] = (e < k) ? lists[(int64_t)row * stride + e] : 0ull;
    __syncwarp();
    for (int g = 1; g < G; ++g) {
        for (int e = lane; e < k; e += 32) mine[k + e] = lists[((int64_t)g * rows + row) * stride + e];
        __syncwarp();
        uint64_t thr;
        warp_prune_list(mine, 2 * k, k, lane, &thr);
        __syncwarp();
    }
    write_topk_row(mine, k, out_s + (int64_t)row * k, out_i + (int64_t)row * k, lane);
    if (Ub || Gb) {  // keys of the tensor-core kernel exclude the per-row user / global bias: add it to the scores now
        float base = Gb ? Gb[0] : 0.f;
        if (Ub) { const int64_t u = u_idx[row]; if (!bad_index(u, n_users)) base += Ub[u]; }
        __syncwarp();
        for (int e = lane; e < k; e += 32) out_s[(int64_t)row * k + e] += base;
    }
}

// ---- merge of G (scores, ids) lists per row: the multi-GPU all-gather merge ----
__global__ void __launch_bounds__(256) topk_merge_pairs_kernel(const float* __restrict__ scores, const int32_t* __restrict__ ids,
                                                               int G, int rows, int k, float* out_s, int32_t* out_i) {
    __shared__ uint64_t buf[8][kCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x * 8 + warp;
    if (row >= rows) return;
    uint64_t* mine = buf[warp];
    for (int e = lane; e < kCap; e += 32) mine[e] = 0ull;
    __syncwarp();
    for (int g = 0; g < G; ++g) {
        const int64_t base = ((int64_t)g * rows + row) * k;
        for (int e = lane; e < k; e += 32) {
            const int32_t id = ids[base + e];
            mine[k + e] = id < 0 ? 0ull : make_key(scores[base + e], (uint32_t)id);
        }
        __syncwarp();
        uint64_t thr;
        warp_prune_list(mine, 2 * k, k, lane, &thr);
        __syncwarp();
    }
    write_topk_row(mine, k, out_s + (int64_t)row * k, out_i + (int64_t)row * k, lane);
}

// ---- top-k of dense logits rows: one warp streams one row ----
__global__ void __launch_bounds__(256) topk_dense_kernel(const float* __restrict__ logits, int rows, int64_t n_cols,
                                                         int64_t row_stride, int k, float* out_s, int32_t* out_i) {
    __shared__ uint64_t buf[8][kCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = blockIdx.x * 8 + warp;
    if (row >= rows) return;
    uint64_t* mine = buf[warp];
    const float* x = logits + (int64_t)row * row_stride;
    int cnt = 0;
    uint64_t thr = 0ull;
    float tauf = -INFINITY;
    for (int64_t c0 = 0; c0 < n_cols; c0 += 128) {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const int64_t c = c0 + h * 32 + lane;
            bool take = false;
            uint64_t key = 0ull;
            if (c < n_cols) {
                const float s = x[c];
                if (s >= tauf) { key = make_key(s, (uint32_t)c); take = key > thr; }
            }
            const unsigned m = __ballot_sync(kFull, take);
            if (take) mine[cnt + __popc(m & ((1u << lane) - 1))] = key;
            cnt += __popc(m);
        }
        __syncwarp();
        if (cnt > kCap - 128) {
            cnt = warp_prune_list(mine, cnt, k, lane, &thr);
            tauf = thr ? key_score(thr) : -INFINITY;
            __syncwarp();
        }
    }
    warp_prune_list(mine, cnt, k, lane, &thr);
    __syncwarp();
    write_topk_row(mine, k, out_s + (int64_t)row * k, out_i + (int64_t)row * k, lane);
}

// ---- ranking metrics (eval/metrics.py:4-105; eval/eval.py:66-99) ----
struct MetricArgs {
    const int32_t* __restrict__ top_ids;   // [Be, k_max]
    const int64_t* __restrict__ u_idx;     // [Be]
    const int64_t* __restrict__ lab_indptr;
    const int32_t* __restrict__ lab_indices;
    const float* __restrict__ y_true;      // dense [Be, n_items] alternative to the CSR
    int64_t n_items;
    const int32_t* __restrict__ user_group;  // [n_users] or null
    const float* __restrict__ discount;    // [k_max] fp32: 1 / log2(r + 2)
    int Be, k_max, n_ks, n_groups;
    int ks[8];
    float* per_user;   // [Be, n_ks, 3] or null   (precision, recall, ndcg)
    double* sums;      // [(1 + n_groups), n_ks, 3]   row 0 = all users
    int64_t* counts;   // [(1 + n_groups)]
};

template <bool DENSE>
__global__ void __launch_bounds__(256) rank_metrics_kernel(MetricArgs a) {
#include "hsk_rank_metrics_body.inc"
}

// ---- trial pack (hsk_eval_topk_pack, hsk_rank_metrics_pack): M models of one shape whose tables are trial 0's + j * stride
// elements.  Kept out of EvalArgs / MetricArgs so that the single-model kernels keep their argument layout.
struct EvalPackArgs {
    int64_t stride;           // elements between two trials' tables
    const int32_t* active;    // [gridDim.z] trial indices
    int n_trials;
    int split_rows;           // n_active * Be: rows of one split's candidate lists, laid out [split][trial][row]
};

// gridDim.z walks the active trials; x / y (row tiles, splits) as the single-model kernel over the shared user batch
__global__ void __launch_bounds__(kEvalThreads, 2) eval_topk_f32_pack_kernel(EvalArgs a, EvalPackArgs pk) {
    {
        const int j = pk.active[blockIdx.z];
        if (j < 0 || j >= pk.n_trials) {
            if (threadIdx.x == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            return;
        }
        const int64_t o = (int64_t)j * pk.stride;
        a.Uw += o; a.Vw += o;
        if (a.Ub) a.Ub += o;
        if (a.Ib) a.Ib += o;
        if (a.Gb) a.Gb += o;
        const int64_t r0 = (int64_t)blockIdx.z * a.Be;   // this trial's first row of the [n_active * Be] outputs
        a.cand += r0 * EV_CAP;
        a.out_scores += r0 * a.k;
        a.out_ids += r0 * a.k;
    }
#define EV_SPLIT_ROWS pk.split_rows
#include "hsk_eval_topk_body.inc"
#undef EV_SPLIT_ROWS
}

struct MetricPackArgs {
    const int32_t* active;    // [gridDim.y] trial indices
    int n_trials;
    int groups;               // the caller's n_groups: trial j's sums / counts start at j * (1 + groups) rows
    int32_t* status;
};

// gridDim.y walks the active trials; x as the single-model kernel over the shared user batch
__global__ void __launch_bounds__(256) rank_metrics_pack_kernel(MetricArgs a, MetricPackArgs pk) {
    constexpr bool DENSE = false;
    {
        const int j = pk.active[blockIdx.y];
        if (j < 0 || j >= pk.n_trials) {
            if (threadIdx.x == 0 && pk.status) atomicOr(pk.status, HSK_STATUS_BAD_INDEX);
            return;
        }
        const int64_t r0 = (int64_t)blockIdx.y * a.Be;
        a.top_ids += r0 * a.k_max;
        if (a.per_user) a.per_user += r0 * a.n_ks * 3;
        a.sums += (int64_t)j * (1 + pk.groups) * a.n_ks * 3;
        a.counts += (int64_t)j * (1 + pk.groups);
    }
#include "hsk_rank_metrics_body.inc"
}

// split plan shared by hsk_eval_topk, hsk_eval_topk_pack and their scratch sizes: a pack multiplies the row tiles by its
// n_active trials, so items are not split where the trials already fill the GPU
static void eval_plan(int Be, int64_t n_local, int n_active, int* n_tiles, int* tiles_per_split, int* n_splits) {
    const int row_tiles = (Be + TM - 1) / TM * n_active;
    const int nt = (int)((n_local + TN - 1) / TN);
    const int want = sm_count() * 2;
    int splits = 1;
    if (row_tiles < want) splits = (want + row_tiles - 1) / row_tiles;
    const int max_splits = nt / 16 > 0 ? nt / 16 : 1;   // at least 16 item tiles per split: every split re-pays the warm-up
                                                        // of its running thresholds (the first ~3 tiles keep everything)
    if (splits > max_splits) splits = max_splits;
    if (splits > 64) splits = 64;
    const int tps = (nt + splits - 1) / splits;
    *n_tiles = nt;
    *tiles_per_split = tps;
    *n_splits = (nt + tps - 1) / tps;
}

int launch_merge_keys(const uint64_t* lists, int n_lists, int rows, int stride, int k, float* out_scores, int32_t* out_ids, cudaStream_t s,
                      const float* Ub, const float* Gb, const int64_t* u_idx, int64_t n_users) {
    topk_merge_keys_kernel<<<(rows + 7) / 8, 256, 0, s>>>(lists, n_lists, rows, stride, k, out_scores, out_ids, Ub, Gb, u_idx, n_users);
    return check_launch("topk merge");
}

}  // namespace hsk

using namespace hsk;

extern "C" int64_t hsk_eval_topk_scratch_bytes(int Be, int64_t n_local_items, int k) {
    (void)k;
    int nt, tps, ns;
    eval_plan(Be > 0 ? Be : 1, n_local_items > 0 ? n_local_items : 1, 1, &nt, &tps, &ns);
    return (int64_t)ns * (Be > 0 ? Be : 1) * EV_CAP * (int64_t)sizeof(uint64_t);
}

extern "C" int hsk_eval_topk(const hsk_mf_tables* t, const int64_t* u_idx, const int64_t* u_rows, int64_t n_users_global,
                             int Be, int64_t id_offset, int64_t id_stride,
                             const int64_t* excl_indptr, const int32_t* excl_indices, int k, float* top_scores,
                             int32_t* top_ids, void* scratch, int64_t scratch_bytes, int32_t* status,
                             hsk_stream_t stream) {
    HSK_REQUIRE(t && t->Uw && t->Vw && u_idx && top_scores && top_ids, "hsk_eval_topk: null pointer");
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && (t->ld % 4) == 0, "hsk_eval_topk: need ld %% 4 == 0 (d=%d ld=%d)", t->d, t->ld);
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw), "hsk_eval_topk: tables must be 16-byte aligned");
    HSK_REQUIRE(k >= 1 && k <= kMaxK, "hsk_eval_topk: 1 <= k <= %d required (k=%d)", kMaxK, k);
    HSK_REQUIRE(t->n_items >= 1 && Be >= 0, "hsk_eval_topk: empty item shard or negative batch");
    HSK_REQUIRE(id_stride >= 1 && id_offset >= 0, "hsk_eval_topk: bad id mapping");
    HSK_REQUIRE((excl_indptr == nullptr) == (excl_indices == nullptr), "hsk_eval_topk: exclusion CSR needs both arrays");
    HSK_REQUIRE(id_offset + (t->n_items - 1) * id_stride < 0x7FFFFFFFll, "hsk_eval_topk: item ids must fit int32");
    if (Be == 0) return HSK_OK;
    EvalArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.u_idx = u_idx; a.u_rows = u_rows; a.excl_indptr = excl_indptr; a.excl_indices = excl_indices;
    a.n_users = u_rows ? n_users_global : t->n_users; a.n_urows = t->n_users; a.n_local = t->n_items; a.id_offset = id_offset; a.id_stride = id_stride;
    a.ld = t->ld; a.Be = Be; a.k = k;
    eval_plan(Be, t->n_items, 1, &a.n_tiles, &a.tiles_per_split, &a.n_splits);
    const int64_t need = (int64_t)a.n_splits * Be * EV_CAP * (int64_t)sizeof(uint64_t);
    HSK_REQUIRE(scratch && scratch_bytes >= need, "hsk_eval_topk: scratch too small (%lld < %lld bytes)",
                (long long)scratch_bytes, (long long)need);
    a.cand = reinterpret_cast<uint64_t*>(scratch);
    a.out_scores = top_scores; a.out_ids = top_ids; a.status = status;
    cudaStream_t s = as_stream(stream);
    dim3 grid((Be + TM - 1) / TM, a.n_splits);
    eval_topk_f32_kernel<<<grid, kEvalThreads, 0, s>>>(a);
    int rc = check_launch("hsk_eval_topk");
    if (rc) return rc;
    if (a.n_splits > 1) rc = launch_merge_keys(a.cand, a.n_splits, Be, EV_CAP, k, top_scores, top_ids, s, nullptr, nullptr, nullptr, 0);
    return rc;
}

static int64_t eval_pack_scratch(int Be, int64_t n_items, int n_active, int* n_tiles, int* tps, int* n_splits) {
    eval_plan(Be, n_items, n_active, n_tiles, tps, n_splits);
    return (int64_t)*n_splits * n_active * Be * EV_CAP * (int64_t)sizeof(uint64_t);
}

extern "C" int64_t hsk_eval_topk_pack_scratch_bytes(int Be, int64_t n_items, int k, int n_active) {
    (void)k;
    int nt, tps, ns;
    return eval_pack_scratch(Be > 0 ? Be : 1, n_items > 0 ? n_items : 1, n_active > 0 ? n_active : 1, &nt, &tps, &ns);
}

extern "C" int hsk_eval_topk_pack(const hsk_mf_tables* t, int64_t trial_stride, int n_trials, const int32_t* active, int n_active,
                                  const int64_t* u_idx, int Be, const int64_t* excl_indptr, const int32_t* excl_indices, int k,
                                  float* top_scores, int32_t* top_ids, void* scratch, int64_t scratch_bytes, int32_t* status,
                                  hsk_stream_t stream) {
    HSK_REQUIRE(t && t->Uw && t->Vw && u_idx && top_scores && top_ids, "hsk_eval_topk_pack: null pointer");
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && (t->ld % 4) == 0, "hsk_eval_topk_pack: need ld %% 4 == 0 (d=%d ld=%d)", t->d, t->ld);
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw), "hsk_eval_topk_pack: tables must be 16-byte aligned");
    HSK_REQUIRE(k >= 1 && k <= kMaxK, "hsk_eval_topk_pack: 1 <= k <= %d required (k=%d)", kMaxK, k);
    HSK_REQUIRE(t->n_items >= 1 && Be >= 0, "hsk_eval_topk_pack: empty item table or negative batch");
    HSK_REQUIRE(t->n_items < 0x7FFFFFFFll, "hsk_eval_topk_pack: item ids must fit int32");
    HSK_REQUIRE((excl_indptr == nullptr) == (excl_indices == nullptr), "hsk_eval_topk_pack: exclusion CSR needs both arrays");
    HSK_REQUIRE(n_trials >= 1 && n_active >= 0 && n_active <= n_trials && n_active <= 65535,
                "hsk_eval_topk_pack: need 0 <= n_active <= n_trials, n_trials >= 1, n_active <= 65535 (n_trials=%d n_active=%d)",
                n_trials, n_active);
    HSK_REQUIRE(n_active == 0 || active, "hsk_eval_topk_pack: active is null");
    HSK_REQUIRE(trial_stride > 0 && trial_stride % 4 == 0,
                "hsk_eval_topk_pack: trial_stride must be a positive multiple of 4 (%lld)", (long long)trial_stride);
    HSK_REQUIRE((int64_t)n_active * Be <= 0x7FFFFFFFll, "hsk_eval_topk_pack: n_active * Be must fit int32");
    if (Be == 0 || n_active == 0) return HSK_OK;
    EvalArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.u_idx = u_idx; a.excl_indptr = excl_indptr; a.excl_indices = excl_indices;
    a.n_users = t->n_users; a.n_urows = t->n_users; a.n_local = t->n_items; a.id_offset = 0; a.id_stride = 1;
    a.ld = t->ld; a.Be = Be; a.k = k;
    const int64_t need = eval_pack_scratch(Be, t->n_items, n_active, &a.n_tiles, &a.tiles_per_split, &a.n_splits);
    HSK_REQUIRE(scratch && scratch_bytes >= need, "hsk_eval_topk_pack: scratch too small (%lld < %lld bytes)",
                (long long)scratch_bytes, (long long)need);
    a.cand = reinterpret_cast<uint64_t*>(scratch);
    a.out_scores = top_scores; a.out_ids = top_ids; a.status = status;
    EvalPackArgs pk;
    pk.stride = trial_stride; pk.active = active; pk.n_trials = n_trials; pk.split_rows = n_active * Be;
    cudaStream_t s = as_stream(stream);
    dim3 grid((Be + TM - 1) / TM, a.n_splits, n_active);
    eval_topk_f32_pack_kernel<<<grid, kEvalThreads, 0, s>>>(a, pk);
    int rc = check_launch("hsk_eval_topk_pack");
    if (rc) return rc;
    // [split][trial][row] lists: one merge over the n_active * Be rows takes every trial's splits
    if (a.n_splits > 1) rc = launch_merge_keys(a.cand, a.n_splits, n_active * Be, EV_CAP, k, top_scores, top_ids, s, nullptr, nullptr, nullptr, 0);
    return rc;
}

extern "C" int hsk_topk_merge(const float* scores, const int32_t* ids, int G, int rows, int k, float* out_scores,
                              int32_t* out_ids, hsk_stream_t stream) {
    HSK_REQUIRE(scores && ids && out_scores && out_ids, "hsk_topk_merge: null pointer");
    HSK_REQUIRE(G >= 1 && rows >= 0 && k >= 1 && k <= kMaxK, "hsk_topk_merge: bad sizes (G=%d rows=%d k=%d)", G, rows, k);
    if (rows == 0) return HSK_OK;
    topk_merge_pairs_kernel<<<(rows + 7) / 8, 256, 0, as_stream(stream)>>>(scores, ids, G, rows, k, out_scores, out_ids);
    return check_launch("hsk_topk_merge");
}

extern "C" int hsk_topk_dense(const float* logits, int rows, int64_t n_cols, int64_t row_stride, int k,
                              float* out_scores, int32_t* out_ids, hsk_stream_t stream) {
    HSK_REQUIRE(logits && out_scores && out_ids, "hsk_topk_dense: null pointer");
    HSK_REQUIRE(k >= 1 && k <= kMaxK, "hsk_topk_dense: 1 <= k <= %d required (k=%d)", kMaxK, k);
    HSK_REQUIRE(n_cols >= k, "hsk_topk_dense: selected index k out of range (k=%d, columns=%lld)", k, (long long)n_cols);
    HSK_REQUIRE(n_cols < 0x7FFFFFFFll && row_stride >= n_cols, "hsk_topk_dense: bad column count / stride");
    if (rows <= 0) return HSK_OK;
    topk_dense_kernel<<<(rows + 7) / 8, 256, 0, as_stream(stream)>>>(logits, rows, n_cols, row_stride, k, out_scores, out_ids);
    return check_launch("hsk_topk_dense");
}

static int metrics_common(MetricArgs& a, const int32_t* top_ids, int Be, int k_max, const int* ks, int n_ks,
                          const int64_t* u_idx, const int32_t* user_group, int n_groups, const float* discount,
                          float* per_user, double* sums, int64_t* counts, const char* who) {
    HSK_REQUIRE(top_ids && ks && u_idx && discount && sums && counts, "%s: null pointer", who);
    HSK_REQUIRE(k_max >= 1 && k_max <= kMaxK && n_ks >= 1 && n_ks <= 8, "%s: need k_max <= %d and at most 8 cut-offs", who, kMaxK);
    for (int i = 0; i < n_ks; ++i) HSK_REQUIRE(ks[i] >= 1 && ks[i] <= k_max, "%s: cut-off %d outside [1, k_max=%d]", who, ks[i], k_max);
    HSK_REQUIRE(n_groups >= 0, "%s: negative group count", who);
    memset(&a, 0, sizeof(a));
    a.top_ids = top_ids; a.u_idx = u_idx; a.user_group = user_group; a.discount = discount;
    a.Be = Be; a.k_max = k_max; a.n_ks = n_ks; a.n_groups = user_group ? n_groups : 0;
    for (int i = 0; i < n_ks; ++i) a.ks[i] = ks[i];
    a.per_user = per_user; a.sums = sums; a.counts = counts;
    return HSK_OK;
}

extern "C" int hsk_rank_metrics(const int32_t* top_ids, int Be, int k_max, const int* ks, int n_ks, const int64_t* u_idx,
                                const int64_t* lab_indptr, const int32_t* lab_indices, const int32_t* user_group,
                                int n_groups, const float* discount, float* per_user, double* sums, int64_t* counts,
                                hsk_stream_t stream) {
    MetricArgs a;
    int rc = metrics_common(a, top_ids, Be, k_max, ks, n_ks, u_idx, user_group, n_groups, discount, per_user, sums, counts,
                            "hsk_rank_metrics");
    if (rc) return rc;
    HSK_REQUIRE(lab_indptr && lab_indices, "hsk_rank_metrics: label CSR is null");
    if (Be <= 0) return HSK_OK;
    a.lab_indptr = lab_indptr; a.lab_indices = lab_indices;
    rank_metrics_kernel<false><<<(Be + 7) / 8, 256, 0, as_stream(stream)>>>(a);
    return check_launch("hsk_rank_metrics");
}

extern "C" int hsk_rank_metrics_dense(const int32_t* top_ids, int Be, int k_max, const int* ks, int n_ks,
                                      const int64_t* u_idx, const float* y_true, int64_t n_items,
                                      const int32_t* user_group, int n_groups, const float* discount, float* per_user,
                                      double* sums, int64_t* counts, hsk_stream_t stream) {
    MetricArgs a;
    int rc = metrics_common(a, top_ids, Be, k_max, ks, n_ks, u_idx, user_group, n_groups, discount, per_user, sums, counts,
                            "hsk_rank_metrics_dense");
    if (rc) return rc;
    HSK_REQUIRE(y_true && n_items >= 1, "hsk_rank_metrics_dense: y_true is null");
    if (Be <= 0) return HSK_OK;
    a.y_true = y_true; a.n_items = n_items;
    rank_metrics_kernel<true><<<(Be + 7) / 8, 256, 0, as_stream(stream)>>>(a);
    return check_launch("hsk_rank_metrics_dense");
}

extern "C" int hsk_rank_metrics_pack(const int32_t* top_ids, int Be, int k_max, const int* ks, int n_ks, const int64_t* u_idx,
                                     const int64_t* lab_indptr, const int32_t* lab_indices, const int32_t* user_group,
                                     int n_groups, const float* discount, int n_trials, const int32_t* active, int n_active,
                                     float* per_user, double* sums, int64_t* counts, int32_t* status, hsk_stream_t stream) {
    MetricArgs a;
    int rc = metrics_common(a, top_ids, Be, k_max, ks, n_ks, u_idx, user_group, n_groups, discount, per_user, sums, counts,
                            "hsk_rank_metrics_pack");
    if (rc) return rc;
    HSK_REQUIRE(lab_indptr && lab_indices, "hsk_rank_metrics_pack: label CSR is null");
    HSK_REQUIRE(n_trials >= 1 && n_active >= 0 && n_active <= n_trials && n_active <= 65535,
                "hsk_rank_metrics_pack: need 0 <= n_active <= n_trials, n_trials >= 1, n_active <= 65535 (n_trials=%d n_active=%d)",
                n_trials, n_active);
    HSK_REQUIRE(n_active == 0 || active, "hsk_rank_metrics_pack: active is null");
    if (Be <= 0 || n_active == 0) return HSK_OK;
    a.lab_indptr = lab_indptr; a.lab_indices = lab_indices;
    MetricPackArgs pk;
    pk.active = active; pk.n_trials = n_trials; pk.groups = n_groups; pk.status = status;
    rank_metrics_pack_kernel<<<dim3((Be + 7) / 8, n_active), 256, 0, as_stream(stream)>>>(a, pk);
    return check_launch("hsk_rank_metrics_pack");
}
