// a1-a7 — the SGD-MF training step's gather / score / loss / scatter kernels (sm_100a).
//
//   hsk_mf_scores          forward only           (algorithms/sgd_alg.py:148-179)
//   hsk_rec_loss           loss + dL/dscores      (train/rec_losses.py:39-139)
//   hsk_mf_scatter_grads   backward of forward    (autograd + embedding_dense_backward in the reference)
//   hsk_mf_train_fused     all of the above in one pass over the gathered rows (train/trainer.py:133-146)
//
// Mapping: one warp owns one gathered row at a time — lane l holds float4 #(l + 32k) of the row (k < NV), so
// every global access is a fully coalesced 128-bit load / 128-bit vector reduction.  A CTA of 4 warps owns one
// sample (user row in registers, item slots strided over the warps); when the batch alone cannot fill the
// machine the item slots are additionally split over gridDim.y (gradients are linear in dL/ds, so partial
// CTAs simply add their share).  All kernels are HBM/L2-bandwidth bound: ~25 issue slots per 16 B moved.
#include <stdlib.h>

#include "hsk_train.cuh"

namespace hsk {

// ------------------------------------------------------------------------------------------------
// forward only
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32) mf_scores_kernel(TrainArgs a, float* __restrict__ scores) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    const int64_t u = a.u_idx[b];
    if (bad_index(u, a.n_users)) {
        if (threadIdx.x == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        return;
    }
    Row<NV> ur;
    ur.load(a.Uw + u * a.ld, a.nvec, lane);
    float bias_u = (a.Ub ? a.Ub[u] : 0.f);
    const float gb = a.Gb ? a.Gb[0] : 0.f;
    const int j0 = blockIdx.y * a.j_per_cta, j1 = min(a.N1, j0 + a.j_per_cta);
    for (int j = j0 + warp; j < j1; j += kWarpsPerCta) {
        const int64_t it = a.i_idx[(int64_t)b * a.N1 + j];
        if (bad_index(it, a.n_items)) {
            if (lane == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        Row<NV> vr;
        vr.load(a.Vw + it * a.ld, a.nvec, lane);
        float s = warp_sum(ur.dot_partial(vr));
        if (lane == 0) {
            // sgd_alg.py:171-178: out = sum(-1); out += u_bias; out += i_bias; out += global_bias
            if (a.Ub) s += bias_u;
            if (a.Ib) s += a.Ib[it];
            if (a.Gb) s += gb;
            scores[(int64_t)b * a.N1 + j] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// loss + dL/dscores from a score matrix: one warp per sample row
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rec_loss_kernel(const float* __restrict__ scores, const double* __restrict__ labels,
                                                       int B, int N1, int kind, float shift, float gscale,
                                                       double* loss_accum, float* __restrict__ dscores,
                                                       float* __restrict__ shifted_out) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    double loss_local = 0.0;
    for (int b = blockIdx.x * wpb + (threadIdx.x >> 5); b < B; b += gridDim.x * wpb) {
        const float* s = scores + (int64_t)b * N1;
        float* ds = dscores ? dscores + (int64_t)b * N1 : nullptr;
        if (kind == HSK_LOSS_BPR) {
            // rec_losses.py:78-86: BCEWithLogits(pos - neg, y) with y = labels[:, 0] (1.0 from the loader)
            const double inv = 1.0 / ((double)B * (double)(N1 - 1));
            const float s0 = s[0];
            const double y = labels ? labels[(int64_t)b * N1] : 1.0;
            float ds0 = 0.f;
            for (int j = 1 + lane; j < N1; j += 32) {
                const float x = s0 - s[j];
                loss_local += ((1.0 - y) * (double)x - (double)log_sigmoid_f(x)) * inv;
                const float dx = (float)(((double)sigmoid_f(x) - y) * inv) * gscale;
                if (ds) ds[j] = -dx;
                ds0 += dx;
            }
            ds0 = warp_sum(ds0);
            if (ds && lane == 0) ds[0] = ds0;
        } else if (kind == HSK_LOSS_SAMPLED_SOFTMAX) {
            // rec_losses.py:131-139: -x0 + logsumexp(x + [j>0]*shift), mean over B
            float mx = -INFINITY;
            for (int j = lane; j < N1; j += 32) mx = fmaxf(mx, s[j] + (j > 0 ? shift : 0.f));
            mx = warp_max(mx);
            float se = 0.f;
            for (int j = lane; j < N1; j += 32) se += expf(s[j] + (j > 0 ? shift : 0.f) - mx);
            se = warp_sum(se);
            const float lse = mx + logf(se);
            const float s0 = s[0];  // read before a possible in-place write of shifted_out
            const float invB = 1.f / (float)B;
            for (int j = lane; j < N1; j += 32) {
                const float x = s[j] + (j > 0 ? shift : 0.f);
                if (ds) ds[j] = (expf(x - lse) - (j == 0 ? 1.f : 0.f)) * invB * gscale;
                if (shifted_out) shifted_out[(int64_t)b * N1 + j] = x;
            }
            if (lane == 0) loss_local += (double)(lse - s0) / (double)B;
        } else {  // HSK_LOSS_BCE, rec_losses.py:39-53: BCEWithLogits over all B*N1 logits
            const double inv = 1.0 / ((double)B * (double)N1);
            for (int j = lane; j < N1; j += 32) {
                const float x = s[j];
                const double y = labels ? labels[(int64_t)b * N1 + j] : (j == 0 ? 1.0 : 0.0);
                loss_local += ((1.0 - y) * (double)x - (double)log_sigmoid_f(x)) * inv;
                if (ds) ds[j] = (float)(((double)sigmoid_f(x) - y) * inv) * gscale;
            }
        }
    }
    loss_local = warp_sum(loss_local);
    __shared__ double red[8];
    if (lane == 0) red[threadIdx.x >> 5] = loss_local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < wpb; ++w) t += red[w];
        if (loss_accum && t != 0.0) atomicAdd(loss_accum, t);
    }
}

// ------------------------------------------------------------------------------------------------
// backward of the forward: scatter-add row gradients given dL/dscores
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32) mf_scatter_kernel(TrainArgs a) {
    __shared__ float4 sm_gu[kWarpsPerCta][NV][32];
    __shared__ float sm_ds[kWarpsPerCta];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    const int64_t u = a.u_idx[b];
    if (bad_index(u, a.n_users)) {
        if (threadIdx.x == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        return;
    }
    Row<NV> ur, gu;
    ur.load(a.Uw + u * a.ld, a.nvec, lane);
    gu.zero();
    float ds_sum = 0.f;
    const int j0 = blockIdx.y * a.j_per_cta, j1 = min(a.N1, j0 + a.j_per_cta);
    for (int j = j0 + warp; j < j1; j += kWarpsPerCta) {
        const int64_t it = a.i_idx[(int64_t)b * a.N1 + j];
        if (bad_index(it, a.n_items)) {
            if (lane == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const float ds = a.dscores_in[(int64_t)b * a.N1 + j];
        Row<NV> vr;
        vr.load(a.Vw + it * a.ld, a.nvec, lane);
        gu.axpy(ds, vr);
        ur.red_scaled(a.gV + it * a.ld, ds, a.nvec, lane);
        if (lane == 0 && a.gIb) atomicAdd(a.gIb + it, ds);
        ds_sum += ds;
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) sm_gu[warp][k][lane] = gu.v[k];
    if (lane == 0) sm_ds[warp] = ds_sum;
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int w = 1; w < kWarpsPerCta; ++w) {
#pragma unroll
            for (int k = 0; k < NV; ++k) {
                float4 o = sm_gu[w][k][lane];
                gu.v[k].x += o.x; gu.v[k].y += o.y; gu.v[k].z += o.z; gu.v[k].w += o.w;
            }
        }
        gu.red(a.gU + u * a.ld, a.nvec, lane);
        if (lane == 0) {
            float t = 0.f;
            for (int w = 0; w < kWarpsPerCta; ++w) t += sm_ds[w];
            if (a.gUb) atomicAdd(a.gUb + u, t);
            if (a.gGb) atomicAdd(a.gGb, t);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// fused forward + loss + backward.  LOSS: 0 bpr, 1 sampled-softmax, 2 bce
// ------------------------------------------------------------------------------------------------
template <int NV, int LOSS>
__global__ void __launch_bounds__(kWarpsPerCta * 32) mf_train_fused_kernel(TrainArgs a) {
#include "hsk_train_fused_body.inc"
}

// trial pack (hsk_mf_train_fused_pack): gridDim.z walks the active trials, gridDim.x / y as the single-model kernel
template <int NV, int LOSS>
__global__ void __launch_bounds__(kWarpsPerCta * 32) mf_train_fused_pack_kernel(TrainArgs a, PackArgs pk) {
    if (!pack_select_trial(a, pk)) return;
#include "hsk_train_fused_body.inc"
}

// ---- host-side argument validation shared by the entry points ----
static int fill_args(TrainArgs& a, const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx,
                     const int64_t* i_idx, int B, int N1, const char* who) {
    HSK_REQUIRE(t && t->Uw && t->Vw, "%s: tables are null", who);
    HSK_REQUIRE(B == 0 || (u_idx && i_idx), "%s: index pointers are null", who);   // an empty batch may come as null
    HSK_REQUIRE(B >= 0 && N1 >= 1, "%s: need B >= 0 and N1 >= 1 (B=%d N1=%d)", who, B, N1);
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && (t->ld % 4) == 0, "%s: need 1 <= d <= ld and ld %% 4 == 0 (d=%d ld=%d)", who,
                t->d, t->ld);
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw), "%s: tables must be 16-byte aligned", who);
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.n_users = t->n_users; a.n_items = t->n_items;
    a.B = B; a.N1 = N1; a.ld = t->ld; a.nvec = t->ld / 4;
    a.u_idx = u_idx; a.i_idx = i_idx;
    if (g) {
        HSK_REQUIRE(g->Uw && g->Vw, "%s: gradient tables are null", who);
        HSK_REQUIRE(g->ld == t->ld && g->d == t->d && g->n_users == t->n_users && g->n_items == t->n_items,
                    "%s: gradient tables must have the layout of the parameter tables", who);
        HSK_REQUIRE(aligned16(g->Uw) && aligned16(g->Vw), "%s: gradient tables must be 16-byte aligned", who);
        HSK_REQUIRE((!t->Ub || g->Ub) && (!t->Ib || g->Ib) && (!t->Gb || g->Gb), "%s: missing bias gradient buffer", who);
        a.gU = g->Uw; a.gV = g->Vw; a.gUb = t->Ub ? g->Ub : nullptr; a.gIb = t->Ib ? g->Ib : nullptr;
        a.gGb = t->Gb ? g->Gb : nullptr;
    }
    return HSK_OK;
}

// item slots per CTA along gridDim.y so that the grid has >= ~8 CTAs per SM when the batch is small
static int pick_j_per_cta(int B, int n_slots, bool splittable) {
    if (!splittable || n_slots <= kWarpsPerCta) return n_slots > 0 ? n_slots : 1;
    const int64_t want_ctas = (int64_t)sm_count() * 8;
    if (B >= want_ctas) return n_slots;
    int64_t splits = (want_ctas + B - 1) / (B > 0 ? B : 1);
    int64_t max_splits = (n_slots + kWarpsPerCta - 1) / kWarpsPerCta;
    if (splits > max_splits) splits = max_splits;
    int per = (int)((n_slots + splits - 1) / splits);
    per = ((per + kWarpsPerCta - 1) / kWarpsPerCta) * kWarpsPerCta;
    return per;
}

}  // namespace hsk

using namespace hsk;

extern "C" int hsk_mf_scores(const hsk_mf_tables* t, const int64_t* u_idx, const int64_t* i_idx, int B, int N1,
                             float* scores, int32_t* status, hsk_stream_t stream) {
    TrainArgs a;
    int rc = fill_args(a, t, nullptr, u_idx, i_idx, B, N1, "hsk_mf_scores");
    if (rc) return rc;
    HSK_REQUIRE(scores, "hsk_mf_scores: scores is null");
    if (B == 0) return HSK_OK;
    a.status = status;
    a.j_per_cta = pick_j_per_cta(B, N1, true);
    dim3 grid(B, (N1 + a.j_per_cta - 1) / a.j_per_cta);
    const int nv = (a.nvec + 31) / 32;
    HSK_DISPATCH_NV(nv, (mf_scores_kernel<NV><<<grid, kWarpsPerCta * 32, 0, as_stream(stream)>>>(a, scores)));
    return check_launch("hsk_mf_scores");
}

extern "C" int hsk_rec_loss(const float* scores, const double* labels, int B, int N1, int loss_kind, float neg_shift,
                            float grad_scale, double* loss_accum, float* dscores, float* shifted_out,
                            hsk_stream_t stream) {
    HSK_REQUIRE(scores, "hsk_rec_loss: scores is null");
    HSK_REQUIRE(B >= 0 && N1 >= 1, "hsk_rec_loss: need B >= 0, N1 >= 1");
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "hsk_rec_loss: unknown loss kind %d", loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "hsk_rec_loss: bpr needs at least one negative");
    if (B == 0) return HSK_OK;
    const int wpb = 8;
    int blocks = (B + wpb - 1) / wpb;
    int cap = sm_count() * 8;
    if (blocks > cap) blocks = cap;
    rec_loss_kernel<<<blocks, wpb * 32, 0, as_stream(stream)>>>(scores, labels, B, N1, loss_kind, neg_shift, grad_scale,
                                                                 loss_accum, dscores, shifted_out);
    return check_launch("hsk_rec_loss");
}

extern "C" int hsk_mf_scatter_grads(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx,
                                    const int64_t* i_idx, const float* dscores, int B, int N1, int32_t* status,
                                    hsk_stream_t stream) {
    TrainArgs a;
    HSK_REQUIRE(g, "hsk_mf_scatter_grads: gradient tables are null");
    int rc = fill_args(a, t, g, u_idx, i_idx, B, N1, "hsk_mf_scatter_grads");
    if (rc) return rc;
    HSK_REQUIRE(dscores, "hsk_mf_scatter_grads: dscores is null");
    if (B == 0) return HSK_OK;
    a.status = status;
    a.dscores_in = dscores;
    a.j_per_cta = pick_j_per_cta(B, N1, true);
    dim3 grid(B, (N1 + a.j_per_cta - 1) / a.j_per_cta);
    const int nv = (a.nvec + 31) / 32;
    HSK_DISPATCH_NV(nv, (mf_scatter_kernel<NV><<<grid, kWarpsPerCta * 32, 0, as_stream(stream)>>>(a)));
    return check_launch("hsk_mf_scatter_grads");
}

extern "C" int hsk_mf_train_fused(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx,
                                  const int64_t* i_idx, int B, int N1, int loss_kind, float neg_shift,
                                  double* loss_accum, float* scores_out, float* dscores_out, int32_t* status,
                                  hsk_stream_t stream) {
    return hsk_mf_train_fused_v(t, g, u_idx, i_idx, B, N1, B, loss_kind, neg_shift, loss_accum, scores_out, dscores_out,
                                status, HSK_TRAIN_AUTO, stream);
}

extern "C" int hsk_mf_train_fused_n(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx,
                                    const int64_t* i_idx, int B, int N1, int64_t B_global, int loss_kind, float neg_shift,
                                    double* loss_accum, float* scores_out, float* dscores_out, int32_t* status,
                                    hsk_stream_t stream) {
    return hsk_mf_train_fused_v(t, g, u_idx, i_idx, B, N1, B_global, loss_kind, neg_shift, loss_accum, scores_out,
                                dscores_out, status, HSK_TRAIN_AUTO, stream);
}

extern "C" int hsk_mf_train_fused_peer(const hsk_mf_tables* t, const hsk_mf_tables* g, const hsk_peer_items* peers,
                                       const int64_t* u_idx, const int64_t* i_idx, int B, int N1, int64_t B_global,
                                       int loss_kind, float neg_shift, double* loss_accum, int64_t step,
                                       const int64_t* step_dev, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(t && g && peers && t->Uw && g->Uw && (B == 0 || (u_idx && i_idx)), "hsk_mf_train_fused_peer: null pointer");
    HSK_REQUIRE(peers->world >= 1 && peers->world <= HSK_MAX_PEERS, "hsk_mf_train_fused_peer: world must be 1..%d", HSK_MAX_PEERS);
    HSK_REQUIRE(B >= 0 && N1 >= 1 && B_global >= B, "hsk_mf_train_fused_peer: bad batch sizes (B=%d N1=%d)", B, N1);
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && (t->ld % 4) == 0 && g->ld == t->ld, "hsk_mf_train_fused_peer: bad row layout");
    HSK_REQUIRE(t->n_items >= 1 && t->n_items < 0x7FFFFFFFll, "hsk_mf_train_fused_peer: the global item count must fit 31 bits");
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "hsk_mf_train_fused_peer: unknown loss kind %d", loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "hsk_mf_train_fused_peer: bpr needs at least one negative");
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(g->Uw), "hsk_mf_train_fused_peer: tables must be 16-byte aligned");
    HSK_REQUIRE((!t->Ub || g->Ub) && (!t->Gb || g->Gb), "hsk_mf_train_fused_peer: missing bias gradient buffer");
    for (int q = 0; q < peers->world; ++q) {
        HSK_REQUIRE(peers->V[q] && peers->gV[q] && aligned16(peers->V[q]) && aligned16(peers->gV[q]),
                    "hsk_mf_train_fused_peer: item tables of rank %d missing or misaligned", q);
        HSK_REQUIRE((peers->Ib[q] != nullptr) == (peers->Ib[0] != nullptr) && (peers->gIb[q] != nullptr) == (peers->Ib[0] != nullptr) &&
                        (peers->stamps[q] != nullptr) == (peers->stamps[0] != nullptr),
                    "hsk_mf_train_fused_peer: item bias / stamps must be set on every rank or on none");
    }
    if (B == 0) return HSK_OK;
    TrainArgs a;
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Ub = t->Ub; a.Gb = t->Gb;
    a.gU = g->Uw; a.gUb = t->Ub ? g->Ub : nullptr; a.gGb = t->Gb ? g->Gb : nullptr;
    a.n_users = t->n_users; a.n_items = t->n_items;
    a.B = B; a.N1 = N1; a.ld = t->ld; a.nvec = t->ld / 4;
    a.u_idx = u_idx; a.i_idx = i_idx;
    a.status = status; a.loss_kind = loss_kind; a.neg_shift = neg_shift; a.loss_accum = loss_accum;
    a.inv_count = loss_kind == HSK_LOSS_BPR ? 1.0 / ((double)B_global * (double)(N1 - 1))
                : loss_kind == HSK_LOSS_BCE ? 1.0 / ((double)B_global * (double)N1) : 1.0 / (double)B_global;
    a.j_per_cta = N1;
    return launch_train_fused_peer(a, *peers, hsk_row_stamp(step), step_dev, loss_kind, as_stream(stream));
}

extern "C" int hsk_mf_train_fused_v(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx,
                                    const int64_t* i_idx, int B, int N1, int64_t B_global, int loss_kind, float neg_shift,
                                    double* loss_accum, float* scores_out, float* dscores_out, int32_t* status,
                                    int variant, hsk_stream_t stream) {
    TrainArgs a;
    HSK_REQUIRE(B_global >= B, "hsk_mf_train_fused_n: the global batch cannot be smaller than the local one");
    HSK_REQUIRE(g, "hsk_mf_train_fused: gradient tables are null");
    HSK_REQUIRE(variant >= HSK_TRAIN_AUTO && variant <= HSK_TRAIN_QWARP, "hsk_mf_train_fused_v: unknown kernel variant %d", variant);
    int rc = fill_args(a, t, g, u_idx, i_idx, B, N1, "hsk_mf_train_fused");
    if (rc) return rc;
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "hsk_mf_train_fused: unknown loss kind %d", loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "hsk_mf_train_fused: bpr needs at least one negative");
    if (B == 0) return HSK_OK;
    a.status = status;
    a.loss_kind = loss_kind;
    a.neg_shift = neg_shift;
    a.loss_accum = loss_accum;
    a.scores_out = scores_out;
    a.dscores_out = dscores_out;
    cudaStream_t s = as_stream(stream);
    const int nv = (a.nvec + 31) / 32;
    const int threads = kWarpsPerCta * 32;
    // Kernel choice (all variants compute the same step; HSK_TRAIN_AUTO picks by shape from the B200 measurements):
    //   quarter-warp kernel (hsk_train_q.cu) for rows <= 128 floats where it measured faster, else for bpr / bce the
    //   bulk-copy ring (hsk_train_tma.cu), else (sampled softmax with long rows) the register-gather kernel of this file
    const bool try_q = variant == HSK_TRAIN_AUTO || variant == HSK_TRAIN_QWARP;
    const bool use_ring = variant != HSK_TRAIN_REGS;
    if (try_q) {
        a.force_q = variant == HSK_TRAIN_QWARP ? 1 : 0;
        a.inv_count = loss_kind == HSK_LOSS_BPR ? 1.0 / ((double)B_global * (double)(N1 - 1))
                    : loss_kind == HSK_LOSS_BCE ? 1.0 / ((double)B_global * (double)N1) : 1.0 / (double)B_global;
        a.j_per_cta = N1;
        const int rcq = launch_train_fused_q(a, loss_kind, s);
        if (rcq != 1) return rcq;
    }
    if (loss_kind == HSK_LOSS_BPR) {
        a.inv_count = 1.0 / ((double)B_global * (double)(N1 - 1));
        a.j_per_cta = pick_j_per_cta(B, N1 - 1, true);
        if (a.j_per_cta > 128) a.j_per_cta = 128;
        dim3 grid(B, (N1 - 1 + a.j_per_cta - 1) / a.j_per_cta);
        if (grid.y > 1 && dscores_out) {  // positive-slot dL/ds is accumulated across gridDim.y
            cudaError_t e = cudaMemsetAsync(dscores_out, 0, sizeof(float) * (size_t)B * N1, s);
            if (e != cudaSuccess) return set_err(HSK_ERR_CUDA, "hsk_mf_train_fused: memset: %s", cudaGetErrorString(e));
        }
        if (use_ring) return launch_train_fused_tma(a, loss_kind, s);
        HSK_DISPATCH_NV(nv, (mf_train_fused_kernel<NV, HSK_LOSS_BPR><<<grid, threads, 0, s>>>(a)));
    } else if (loss_kind == HSK_LOSS_BCE) {
        a.inv_count = 1.0 / ((double)B_global * (double)N1);
        a.j_per_cta = pick_j_per_cta(B, N1, true);
        if (a.j_per_cta > 128) a.j_per_cta = 128;
        dim3 grid(B, (N1 + a.j_per_cta - 1) / a.j_per_cta);
        if (use_ring) return launch_train_fused_tma(a, loss_kind, s);
        HSK_DISPATCH_NV(nv, (mf_train_fused_kernel<NV, HSK_LOSS_BCE><<<grid, threads, 0, s>>>(a)));
    } else {
        a.inv_count = 1.0 / (double)B_global;
        a.j_per_cta = N1;
        dim3 grid(B, 1);
        const size_t smem = sizeof(float) * (size_t)N1;
        HSK_REQUIRE(smem <= 40 * 1024, "hsk_mf_train_fused: sampled-softmax supports at most 10240 slots per sample");
        HSK_DISPATCH_NV(nv, (mf_train_fused_kernel<NV, HSK_LOSS_SAMPLED_SOFTMAX><<<grid, threads, smem, s>>>(a)));
    }
    return check_launch("hsk_mf_train_fused");
}

extern "C" int hsk_mf_train_fused_pack(const hsk_mf_tables* t, const hsk_mf_tables* g, int64_t trial_stride, int n_trials,
                                       const int32_t* active, int n_active, const int64_t* u_idx, const int64_t* i_idx, int B,
                                       int N1, int loss_kind, float neg_shift, double* loss_accum, int32_t* status,
                                       hsk_stream_t stream) {
    TrainArgs a;
    HSK_REQUIRE(g, "hsk_mf_train_fused_pack: gradient tables are null");
    int rc = fill_args(a, t, g, u_idx, i_idx, B, N1, "hsk_mf_train_fused_pack");
    if (rc) return rc;
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "hsk_mf_train_fused_pack: unknown loss kind %d", loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "hsk_mf_train_fused_pack: bpr needs at least one negative");
    HSK_REQUIRE(n_trials >= 1 && n_active >= 0 && n_active <= n_trials && n_active <= 65535,
                "hsk_mf_train_fused_pack: need 0 <= n_active <= n_trials, n_trials >= 1, n_active <= 65535 (n_trials=%d n_active=%d)",
                n_trials, n_active);
    HSK_REQUIRE(n_active == 0 || active, "hsk_mf_train_fused_pack: active is null");
    HSK_REQUIRE(trial_stride > 0 && trial_stride % 4 == 0,
                "hsk_mf_train_fused_pack: trial_stride must be a positive multiple of 4 (%lld)", (long long)trial_stride);
    if (B == 0 || n_active == 0) return HSK_OK;
    a.status = status;
    a.loss_kind = loss_kind;
    a.neg_shift = neg_shift;
    a.loss_accum = loss_accum;
    a.inv_count = loss_kind == HSK_LOSS_BPR ? 1.0 / ((double)B * (double)(N1 - 1))
                : loss_kind == HSK_LOSS_BCE ? 1.0 / ((double)B * (double)N1) : 1.0 / (double)B;
    PackArgs pk;
    pk.stride = trial_stride;
    pk.active = active;
    pk.n_trials = n_trials;
    cudaStream_t s = as_stream(stream);
    // HSK_TRAIN_AUTO's rules applied to the work of the whole launch (n_active * B samples); where AUTO would take the
    // bulk-copy ring, the register-gather kernel runs instead (the ring is not packed)
    const int64_t work = (int64_t)n_active * B;
    if (train_fused_q_fits(work, a.nvec, N1, loss_kind, false)) {
        a.j_per_cta = N1;
        return launch_train_fused_q_pack(a, pk, n_active, loss_kind, s);
    }
    const int work_i = work < 0x7FFFFFFF ? (int)work : 0x7FFFFFFF;
    const int nv = (a.nvec + 31) / 32;
    const int threads = kWarpsPerCta * 32;
    if (loss_kind == HSK_LOSS_BPR) {
        a.j_per_cta = pick_j_per_cta(work_i, N1 - 1, true);
        if (a.j_per_cta > 128) a.j_per_cta = 128;
        dim3 grid(B, (N1 - 1 + a.j_per_cta - 1) / a.j_per_cta, n_active);
        HSK_DISPATCH_NV(nv, (mf_train_fused_pack_kernel<NV, HSK_LOSS_BPR><<<grid, threads, 0, s>>>(a, pk)));
    } else if (loss_kind == HSK_LOSS_BCE) {
        a.j_per_cta = pick_j_per_cta(work_i, N1, true);
        if (a.j_per_cta > 128) a.j_per_cta = 128;
        dim3 grid(B, (N1 + a.j_per_cta - 1) / a.j_per_cta, n_active);
        HSK_DISPATCH_NV(nv, (mf_train_fused_pack_kernel<NV, HSK_LOSS_BCE><<<grid, threads, 0, s>>>(a, pk)));
    } else {
        a.j_per_cta = N1;
        dim3 grid(B, 1, n_active);
        const size_t smem = sizeof(float) * (size_t)N1;
        HSK_REQUIRE(smem <= 40 * 1024, "hsk_mf_train_fused_pack: sampled-softmax supports at most 10240 slots per sample");
        HSK_DISPATCH_NV(nv, (mf_train_fused_pack_kernel<NV, HSK_LOSS_SAMPLED_SOFTMAX><<<grid, threads, smem, s>>>(a, pk)));
    }
    return check_launch("hsk_mf_train_fused_pack");
}

// ---- row gather / scatter-add used by the item-sharded step (hassaku_b200/sharded.py): the rows a peer asked for are
// packed contiguously before the all-to-all, and the row gradients received back are added into the owner's table ----
namespace hsk {
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ src, int ld, const int64_t* __restrict__ idx,
                                                          int64_t n, int64_t n_src, float* __restrict__ dst, int32_t* status) {
    const int nvec = ld >> 2;
    const int lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < n; r += (int64_t)gridDim.x * 8) {
        const int64_t s = idx[r];
        if (bad_index(s, n_src)) {
            if (lane == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const float4* sp = reinterpret_cast<const float4*>(src + s * ld);
        float4* dp = reinterpret_cast<float4*>(dst + r * ld);
        for (int k = lane; k < nvec; k += 32) dp[k] = __ldg(sp + k);
    }
}
__global__ void __launch_bounds__(256) scatter_add_rows_kernel(float* __restrict__ dst, int ld, const int64_t* __restrict__ idx,
                                                               int64_t n, int64_t n_dst, const float* __restrict__ src, int32_t* status) {
    const int nvec = ld >> 2;
    const int lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < n; r += (int64_t)gridDim.x * 8) {
        const int64_t d = idx[r];
        if (bad_index(d, n_dst)) {
            if (lane == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const float4* sp = reinterpret_cast<const float4*>(src + r * ld);
        float4* dp = reinterpret_cast<float4*>(dst + d * ld);
        for (int k = lane; k < nvec; k += 32) atomicAdd(dp + k, sp[k]);
    }
}
}  // namespace hsk

static int rows_args_ok(const float* a, const float* b, int ld, const int64_t* idx, const char* who) {
    HSK_REQUIRE(a && b && idx, "%s: null pointer", who);
    HSK_REQUIRE(ld >= 4 && (ld % 4) == 0 && aligned16(a) && aligned16(b), "%s: rows must be 16-byte aligned with ld %% 4 == 0", who);
    return HSK_OK;
}

extern "C" int hsk_gather_rows(const float* src, int ld, const int64_t* idx, int64_t n, int64_t n_src, float* dst,
                               int32_t* status, hsk_stream_t stream) {
    int rc = rows_args_ok(src, dst, ld, idx, "hsk_gather_rows");
    if (rc) return rc;
    if (n <= 0) return HSK_OK;
    int64_t blocks = (n + 7) / 8, cap = (int64_t)sm_count() * 16;
    gather_rows_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(src, ld, idx, n, n_src, dst, status);
    return check_launch("hsk_gather_rows");
}

extern "C" int hsk_scatter_add_rows(float* dst, int ld, const int64_t* idx, int64_t n, int64_t n_dst, const float* src,
                                    int32_t* status, hsk_stream_t stream) {
    int rc = rows_args_ok(dst, src, ld, idx, "hsk_scatter_add_rows");
    if (rc) return rc;
    if (n <= 0) return HSK_OK;
    int64_t blocks = (n + 7) / 8, cap = (int64_t)sm_count() * 16;
    scatter_add_rows_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(dst, ld, idx, n, n_dst, src, status);
    return check_launch("hsk_scatter_add_rows");
}

namespace hsk {
__global__ void __launch_bounds__(256) shard_local_index_kernel(const int64_t* __restrict__ idx, int64_t n, int world,
                                                                int64_t rank_stride, int64_t* __restrict__ out) {
    for (int64_t e = blockIdx.x * 256ll + threadIdx.x; e < n; e += (int64_t)gridDim.x * 256) {
        const int64_t i = idx[e];
        out[e] = i < 0 ? i : (i % world) * rank_stride + i / world;
    }
}
}  // namespace hsk

extern "C" int hsk_shard_local_index(const int64_t* idx, int64_t n, int world, int64_t rank_stride, int64_t* out,
                                     hsk_stream_t stream) {
    HSK_REQUIRE(n >= 0 && world >= 1 && rank_stride >= 0, "hsk_shard_local_index: bad sizes");
    if (n == 0) return HSK_OK;
    HSK_REQUIRE(idx && out, "hsk_shard_local_index: null pointer");
    const int64_t blocks = (n + 255) / 256, cap = (int64_t)sm_count() * 8;
    shard_local_index_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(idx, n, world, rank_stride, out);
    return check_launch("hsk_shard_local_index");
}
