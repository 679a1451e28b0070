// fp32 re-scoring of the tensor-core evaluator's candidates (north_star: TF32 / BF16 mode with top-k recall overlap
// >= 0.999 against the fp32 path of eval/eval.py:243-253).
//
// The tcgen05 kernel ranks all items with bf16 / tf32 operands and hands over its best n_cand > k candidates per user
// (exclusions already removed).  Here every candidate is scored again from the fp32 tables — a warp per user keeps the
// user row in registers, streams the n_cand item rows with coalesced 128-bit loads (4 rows in flight), reduces by
// shuffle — and the exact top-k of the candidates is selected with the 64-bit (score, id) keys of hsk_topk.cuh, so the
// order rule (score descending, lower id first) and the score values are those of the fp32 evaluator.  A true top-k item
// can only be missed if the low-precision pass ranked it below n_cand: with n_cand = k + 28 that needs a score error
// 28 ranks wide (measured overlap 1.0 on the test distributions).
// Cost: n_cand rows of 4 d bytes per user (cfg5: 128 KB / user, ~6 % of the scoring time at 1 M items).
#include "hsk_topk.cuh"

namespace hsk {

constexpr int kRescoreMax = 128;   // candidates per user: 4 keys per lane
constexpr int kRescoreKPL = kRescoreMax / 32;

struct RescoreArgs {
    const float* __restrict__ Uw;
    const float* __restrict__ Vw;
    const float* __restrict__ Ub;
    const float* __restrict__ Ib;
    const float* __restrict__ Gb;
    const int64_t* __restrict__ u_idx;    // row of Uw / Ub per batch entry
    const int32_t* __restrict__ cand;     // [Be, n_cand] global item ids, < 0 = empty
    const float* __restrict__ cand_scores;   // [Be, n_cand] or null: -inf marks an EXCLUDED item (stays -inf)
    int64_t n_users, n_local, id_offset, id_stride;
    int Be, n_cand, k, ld, nvec;
    float* out_scores;
    int32_t* out_ids;
    int32_t* status;
    // item tables sharded over the ranks of a node and mapped here (hsk_rescore_topk_shards): item id = q + n_shards * row of
    // shard q; n_shards <= 1: the one table Vw / Ib with the id_offset / id_stride mapping
    int n_shards;
    const float* shard_V[HSK_MAX_PEERS];
    const float* shard_Ib[HSK_MAX_PEERS];
    int64_t shard_rows[HSK_MAX_PEERS];
};

// POSITIONAL (item-sharded evaluation): no selection — out_scores[row, c] = the fp32 score of candidate c if THIS shard owns
// it ((id - id_offset) % id_stride == 0), else -inf; ids of other shards are expected and not reported.
template <int NV, bool POSITIONAL>
__global__ void __launch_bounds__(256) rescore_topk_kernel(RescoreArgs a) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= a.Be) return;
    const int64_t u = a.u_idx[row];
    float* os = a.out_scores + (int64_t)row * (POSITIONAL ? a.n_cand : a.k);
    int32_t* oi = POSITIONAL ? nullptr : a.out_ids + (int64_t)row * a.k;
    if (bad_index(u, a.n_users)) {
        if (lane == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        for (int e = lane; e < (POSITIONAL ? a.n_cand : a.k); e += 32) { os[e] = -INFINITY; if (!POSITIONAL) oi[e] = -1; }
        return;
    }
    Row<NV> ur;
    ur.load(a.Uw + u * a.ld, a.nvec, lane);
    const float base = (a.Ub ? a.Ub[u] : 0.f) + (a.Gb ? a.Gb[0] : 0.f);
    const int32_t* cand = a.cand + (int64_t)row * a.n_cand;
    uint64_t key[kRescoreKPL];
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) key[r] = 0ull;
    // lane l looks up candidate r * 32 + l: id -> local row (id = id_offset + local * id_stride)
    int64_t loc[kRescoreKPL];
    int32_t gid[kRescoreKPL];
    int own[kRescoreKPL];
    bool masked[kRescoreKPL];
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) {
        const int c = r * 32 + lane;
        gid[r] = (c < a.n_cand) ? cand[c] : -1;
        // an item of the user's exclusion row that surfaced because fewer than n_cand admissible items exist: the
        // low-precision pass reports it with score -inf, and -inf it stays (eval/eval.py:250-251)
        masked[r] = a.cand_scores && c < a.n_cand && a.cand_scores[(int64_t)row * a.n_cand + c] == -INFINITY;
        loc[r] = -1;
        own[r] = 0;
        if (gid[r] >= 0 && a.n_shards > 1) {
            const int q = gid[r] % a.n_shards;
            const int64_t l = gid[r] / a.n_shards;
            if (l >= a.shard_rows[q]) {
                if (a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
                gid[r] = -1;
            } else {
                loc[r] = l;
                own[r] = q;
            }
        } else if (gid[r] >= 0) {
            const int64_t rel = (int64_t)gid[r] - a.id_offset;
            const int64_t l = rel / a.id_stride;
            if (rel < 0 || l * a.id_stride != rel || l >= a.n_local) {
                if (!POSITIONAL && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
                gid[r] = -1;
            } else {
                loc[r] = l;
            }
        }
    }
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) {
        if (r * 32 >= a.n_cand) break;
        float sc = 0.f;   // lane j ends up holding the score of candidate r * 32 + j
#pragma unroll 1
        for (int j0 = 0; j0 < 32; j0 += 4) {
            int64_t l[4];
            Row<NV> vr[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                l[q] = __shfl_sync(kFull, loc[r], j0 + q);
                const int oq = __shfl_sync(kFull, own[r], j0 + q);
                const float* vb = a.n_shards > 1 ? a.shard_V[oq] : a.Vw;
                if (l[q] >= 0) vr[q].load(vb + l[q] * a.ld, a.nvec, lane); else vr[q].zero();
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float s = warp_sum(ur.dot_partial(vr[q]));
                if (lane == j0 + q) sc = s;
            }
        }
        if (loc[r] >= 0) {
            const float* ibq = a.n_shards > 1 ? a.shard_Ib[own[r]] : a.Ib;
            if (ibq) sc += __ldg(ibq + loc[r]);
            key[r] = make_key(masked[r] ? -INFINITY : sc, (uint32_t)gid[r]);
        }
        if (POSITIONAL) {
            const int c = r * 32 + lane;
            if (c < a.n_cand) os[c] = (loc[r] >= 0 && !masked[r]) ? sc + base : -INFINITY;
        }
    }
    if (POSITIONAL) return;
    warp_sort_desc<kRescoreKPL>(key, lane);
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) {
        const int e = r * 32 + lane;
        if (e < a.k) {
            const float sc = key[r] ? key_score(key[r]) : -INFINITY;
            os[e] = sc == -INFINITY ? sc : sc + base;
            oi[e] = key_id(key[r]);
        }
    }
}

}  // namespace hsk

using namespace hsk;

extern "C" int hsk_rescore_topk(const hsk_mf_tables* t, const int64_t* u_rows, int Be, int64_t id_offset, int64_t id_stride,
                                const int32_t* cand_ids, const float* cand_scores, int n_cand, int k, float* top_scores,
                                int32_t* top_ids, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(t && t->Uw && t->Vw && u_rows && cand_ids && top_scores && top_ids, "hsk_rescore_topk: null pointer");
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && t->ld % 4 == 0 && t->ld <= 1024, "hsk_rescore_topk: bad table shape");
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw), "hsk_rescore_topk: tables must be 16-byte aligned");
    HSK_REQUIRE(n_cand >= 1 && n_cand <= kRescoreMax && k >= 1 && k <= n_cand, "hsk_rescore_topk: need 1 <= k <= n_cand <= %d", kRescoreMax);
    HSK_REQUIRE(id_stride >= 1 && id_offset >= 0 && Be >= 0, "hsk_rescore_topk: bad id mapping / batch");
    if (Be == 0) return HSK_OK;
    RescoreArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.u_idx = u_rows; a.cand = cand_ids; a.cand_scores = cand_scores;
    a.n_users = t->n_users; a.n_local = t->n_items; a.id_offset = id_offset; a.id_stride = id_stride;
    a.Be = Be; a.n_cand = n_cand; a.k = k; a.ld = t->ld; a.nvec = t->ld / 4;
    a.out_scores = top_scores; a.out_ids = top_ids; a.status = status;
    const int nv = (a.nvec + 31) / 32;
    const int blocks = (Be + 7) / 8;
    cudaStream_t s = as_stream(stream);
    HSK_DISPATCH_NV(nv, (rescore_topk_kernel<NV, false><<<blocks, 256, 0, s>>>(a)));
    return check_launch("hsk_rescore_topk");
}

extern "C" int hsk_rescore_topk_shards(const hsk_mf_tables* t, const float* const* V_shards, const int64_t* shard_rows,
                                       const float* const* Ib_shards, int n_shards, const int64_t* u_rows, int Be,
                                       const int32_t* cand_ids, const float* cand_scores, int n_cand, int k, float* top_scores,
                                       int32_t* top_ids, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(t && t->Uw && V_shards && shard_rows && u_rows && cand_ids && top_scores && top_ids, "hsk_rescore_topk_shards: null pointer");
    HSK_REQUIRE(n_shards >= 1 && n_shards <= HSK_MAX_PEERS, "hsk_rescore_topk_shards: 1..%d shards", HSK_MAX_PEERS);
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && t->ld % 4 == 0 && t->ld <= 1024 && aligned16(t->Uw), "hsk_rescore_topk_shards: bad table shape");
    HSK_REQUIRE(n_cand >= 1 && n_cand <= kRescoreMax && k >= 1 && k <= n_cand && Be >= 0, "hsk_rescore_topk_shards: need 1 <= k <= n_cand <= %d", kRescoreMax);
    if (Be == 0) return HSK_OK;
    RescoreArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Ub = t->Ub; a.Gb = t->Gb;
    a.u_idx = u_rows; a.cand = cand_ids; a.cand_scores = cand_scores;
    a.n_users = t->n_users; a.id_offset = 0; a.id_stride = 1;
    a.Be = Be; a.n_cand = n_cand; a.k = k; a.ld = t->ld; a.nvec = t->ld / 4;
    a.out_scores = top_scores; a.out_ids = top_ids; a.status = status;
    // the kernel's shard path is taken for n_shards > 1; one shard = the plain mapping on that table
    a.n_shards = n_shards;
    for (int q = 0; q < n_shards; ++q) {
        HSK_REQUIRE(V_shards[q] && aligned16(V_shards[q]) && shard_rows[q] >= 1, "hsk_rescore_topk_shards: table of shard %d missing, misaligned or empty", q);
        a.shard_V[q] = V_shards[q];
        a.shard_Ib[q] = Ib_shards ? Ib_shards[q] : nullptr;
        a.shard_rows[q] = shard_rows[q];
    }
    a.Vw = V_shards[0]; a.Ib = Ib_shards ? Ib_shards[0] : nullptr; a.n_local = shard_rows[0];
    const int nv = (a.nvec + 31) / 32;
    const int blocks = (Be + 7) / 8;
    cudaStream_t s = as_stream(stream);
    HSK_DISPATCH_NV(nv, (rescore_topk_kernel<NV, false><<<blocks, 256, 0, s>>>(a)));
    return check_launch("hsk_rescore_topk_shards");
}

extern "C" int hsk_rescore_scores(const hsk_mf_tables* t, const int64_t* u_rows, int Be, int64_t id_offset, int64_t id_stride,
                                  const int32_t* cand_ids, int n_cand, float* out_scores, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(t && t->Uw && t->Vw && u_rows && cand_ids && out_scores, "hsk_rescore_scores: null pointer");
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && t->ld % 4 == 0 && t->ld <= 1024, "hsk_rescore_scores: bad table shape");
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw), "hsk_rescore_scores: tables must be 16-byte aligned");
    HSK_REQUIRE(n_cand >= 1 && n_cand <= kRescoreMax, "hsk_rescore_scores: need 1 <= n_cand <= %d", kRescoreMax);
    HSK_REQUIRE(id_stride >= 1 && id_offset >= 0 && Be >= 0, "hsk_rescore_scores: bad id mapping / batch");
    if (Be == 0) return HSK_OK;
    RescoreArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.u_idx = u_rows; a.cand = cand_ids;
    a.n_users = t->n_users; a.n_local = t->n_items; a.id_offset = id_offset; a.id_stride = id_stride;
    a.Be = Be; a.n_cand = n_cand; a.k = n_cand; a.ld = t->ld; a.nvec = t->ld / 4;
    a.out_scores = out_scores; a.status = status;
    const int nv = (a.nvec + 31) / 32;
    const int blocks = (Be + 7) / 8;
    cudaStream_t s = as_stream(stream);
    HSK_DISPATCH_NV(nv, (rescore_topk_kernel<NV, true><<<blocks, 256, 0, s>>>(a)));
    return check_launch("hsk_rescore_scores");
}

// ---- item-sharded evaluation, last step: the owner of a user row holds the merged candidate ids [rows, n_cand] and, from
// every shard, the positional fp32 scores [G, rows, n_cand] (finite only where that shard owns the item): the score of a
// candidate is the maximum over the shards; the k best by (score desc, id asc) are the row's result.  A candidate whose
// merged low-precision score (cand_scores, nullable) is -inf is an excluded item of the row's -inf tail: it stays -inf.
namespace hsk {
__global__ void __launch_bounds__(256) topk_combine_kernel(const float* __restrict__ scores, const int32_t* __restrict__ ids,
                                                           const float* __restrict__ cand_scores, int G,
                                                           int rows, int n_cand, int k, float* __restrict__ out_s,
                                                           int32_t* __restrict__ out_i) {
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= rows) return;
    uint64_t key[kRescoreKPL];
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) {
        const int c = r * 32 + lane;
        key[r] = 0ull;
        if (c < n_cand) {
            const int32_t id = ids[(int64_t)row * n_cand + c];
            if (id >= 0) {
                float sc = -INFINITY;
                if (!cand_scores || cand_scores[(int64_t)row * n_cand + c] != -INFINITY)
                    for (int q = 0; q < G; ++q) sc = fmaxf(sc, scores[((int64_t)q * rows + row) * n_cand + c]);
                key[r] = make_key(sc, (uint32_t)id);
            }
        }
    }
    warp_sort_desc<kRescoreKPL>(key, lane);
#pragma unroll
    for (int r = 0; r < kRescoreKPL; ++r) {
        const int e = r * 32 + lane;
        if (e < k) {
            out_s[(int64_t)row * k + e] = key[r] ? key_score(key[r]) : -INFINITY;
            out_i[(int64_t)row * k + e] = key_id(key[r]);
        }
    }
}
}  // namespace hsk

extern "C" int hsk_topk_combine(const float* scores, const int32_t* ids, const float* cand_scores, int G, int rows, int n_cand,
                                int k, float* out_scores, int32_t* out_ids, hsk_stream_t stream) {
    HSK_REQUIRE(scores && ids && out_scores && out_ids, "hsk_topk_combine: null pointer");
    HSK_REQUIRE(G >= 1 && rows >= 0 && n_cand >= 1 && n_cand <= kRescoreMax && k >= 1 && k <= n_cand, "hsk_topk_combine: bad sizes");
    if (rows == 0) return HSK_OK;
    topk_combine_kernel<<<(rows + 7) / 8, 256, 0, as_stream(stream)>>>(scores, ids, cand_scores, G, rows, n_cand, k, out_scores, out_ids);
    return check_launch("hsk_topk_combine");
}
