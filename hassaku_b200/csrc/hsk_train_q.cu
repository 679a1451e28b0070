// hsk_mf_train_fused for SMALL rows (ld <= 128 floats, i.e. embedding_dim <= 128): quarter-warp-per-sample kernel.
//
// Why a second layout: with d = 128 a row is one float4 per lane of a warp, so the warp-per-row kernels
// (hsk_train.cu, hsk_train_tma.cu) spend ~100 warp instructions of fixed cost per row (5-step shuffle reduction, index
// broadcast, address arithmetic, loss math, barrier bookkeeping) around 4 FMAs of payload and are ISSUE bound
// (ncu r01: 57 % issue-slot utilisation at 25 % occupancy on the cfg3 shape), not memory bound.
// Here 8 lanes own one SAMPLE: each lane holds 4 float4 (16 floats) of the user row and of the dL/du accumulator, a row
// dot product needs 3 shuffle steps instead of 5, and every warp instruction works on 4 samples at once, so the fixed
// cost per row drops ~4x.  A group walks its sample's N1 item rows 4 at a time (16 independent 16-byte loads in flight
// per lane), nothing is shared between groups: no shared-memory staging, no block barrier (sampled softmax keeps its
// shifted scores in a per-group strip of shared memory, synchronised with __syncwarp only).
// A quarter-warp reading 128 contiguous bytes per 16-byte-per-lane load is exactly one fully used 128-byte line.
#include "hsk_train.cuh"

namespace hsk {

constexpr int kQWarps = 2;            // warps per CTA -> 8 samples per CTA
constexpr int kQUnroll = 4;           // item rows of a sample in flight per group

template <int K4>
struct QRow {
    float4 v[K4];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int k = 0; k < K4; ++k) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // lane l of the group holds float4 l + 8 k; only the last k can run past the row
    __device__ __forceinline__ void load(const float* __restrict__ row, int l, bool last_ok) {
        const float4* p = reinterpret_cast<const float4*>(row) + l;
#pragma unroll
        for (int k = 0; k < K4; ++k) v[k] = (k < K4 - 1 || last_ok) ? __ldg(p + 8 * k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // a row that may live in a PEER's memory (NVLink): ordinary coherent loads, not the read-only path
    __device__ __forceinline__ void load_peer(const float* row, int l, bool last_ok) {
        const float4* p = reinterpret_cast<const float4*>(row) + l;
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            if (k < K4 - 1 || last_ok) {
                asm volatile("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];\n"
                             : "=f"(v[k].x), "=f"(v[k].y), "=f"(v[k].z), "=f"(v[k].w) : "l"(p + 8 * k) : "memory");
            } else {
                v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    }
    __device__ __forceinline__ float dot(const QRow& o) const {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            a0 = fmaf(v[k].x, o.v[k].x, a0);
            a1 = fmaf(v[k].y, o.v[k].y, a1);
            a0 = fmaf(v[k].z, o.v[k].z, a0);
            a1 = fmaf(v[k].w, o.v[k].w, a1);
        }
        return a0 + a1;
    }
    __device__ __forceinline__ void axpy(float a, const QRow& o) {
#pragma unroll
        for (int k = 0; k < K4; ++k) {
            v[k].x = fmaf(a, o.v[k].x, v[k].x);
            v[k].y = fmaf(a, o.v[k].y, v[k].y);
            v[k].z = fmaf(a, o.v[k].z, v[k].z);
            v[k].w = fmaf(a, o.v[k].w, v[k].w);
        }
    }
    // dst += a * this  (RED.E.ADD.F32x4)
    __device__ __forceinline__ void red(float* dst, float a, int l, bool last_ok) const {
        float4* p = reinterpret_cast<float4*>(dst) + l;
#pragma unroll
        for (int k = 0; k < K4; ++k)
            if (k < K4 - 1 || last_ok) atomicAdd(p + 8 * k, make_float4(a * v[k].x, a * v[k].y, a * v[k].z, a * v[k].w));
    }
    // the same into a peer's gradient table: system scope — the addition is performed in the OWNER's L2, atomically with the
    // other ranks' and the owner's own contributions
    __device__ __forceinline__ void red_peer(float* dst, float a, int l, bool last_ok) const {
        float4* p = reinterpret_cast<float4*>(dst) + l;
#if defined(HSK_MEASURE_PEER_NORED)      // measurement builds only (profiles/r02_peer_exchange.md): what the reductions cost on the link
        (void)p;
#elif defined(HSK_MEASURE_PEER_STORE)    // ... and what the same bytes cost as plain stores (WRONG results)
#pragma unroll
        for (int k = 0; k < K4; ++k)
            if (k < K4 - 1 || last_ok) p[8 * k] = make_float4(a * v[k].x, a * v[k].y, a * v[k].z, a * v[k].w);
#else
#pragma unroll
        for (int k = 0; k < K4; ++k)
            if (k < K4 - 1 || last_ok)
                asm volatile("red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" ::"l"(p + 8 * k), "f"(a * v[k].x),
                             "f"(a * v[k].y), "f"(a * v[k].z), "f"(a * v[k].w)
                             : "memory");
#endif
    }
};

__device__ __forceinline__ float group_sum(float v) {   // over the 8 lanes of a quarter-warp; every lane gets the sum
    v += __shfl_xor_sync(kFull, v, 4);
    v += __shfl_xor_sync(kFull, v, 2);
    v += __shfl_xor_sync(kFull, v, 1);
    return v;
}
__device__ __forceinline__ float group_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(kFull, v, 4));
    v = fmaxf(v, __shfl_xor_sync(kFull, v, 2));
    v = fmaxf(v, __shfl_xor_sync(kFull, v, 1));
    return v;
}

// PEER mode (hsk_mf_train_fused_peer): the item tables are sharded over the ranks of a node, item i = row i / world of rank
// i % world, every rank's shard mapped into this address space
struct PeerArgs {
    hsk_peer_items p;
    int lg;                 // log2(world) when world is a power of two, else -1
    int stamp_host;
    const int64_t* step_dev;
};
struct ItemAt {             // where one item's row / bias / gradients / stamp live
    const float* v;
    float* g;
    const float* ib;
    float* gib;
    uint8_t* st;
};
template <bool PEER>
__device__ __forceinline__ ItemAt item_at(const TrainArgs& a, const PeerArgs& pv, int64_t it, int ld) {
    ItemAt x;
    if (!PEER) {
        x.v = a.Vw + it * ld; x.g = a.gV + it * ld; x.ib = a.Ib ? a.Ib + it : nullptr; x.gib = a.gIb ? a.gIb + it : nullptr;
        x.st = nullptr;
        return x;
    }
    const uint32_t i = (uint32_t)it;            // global item ids < 2^31 (checked at launch)
    uint32_t own, row;
    if (pv.lg >= 0) { own = i & ((1u << pv.lg) - 1u); row = i >> pv.lg; }
    else { row = i / (uint32_t)pv.p.world; own = i - row * (uint32_t)pv.p.world; }
    const int64_t off = (int64_t)row * ld;
    x.v = pv.p.V[own] + off; x.g = pv.p.gV[own] + off;
    x.ib = pv.p.Ib[own] ? pv.p.Ib[own] + row : nullptr;
    x.gib = pv.p.gIb[own] ? pv.p.gIb[own] + row : nullptr;
    x.st = pv.p.stamps[own] ? pv.p.stamps[own] + row : nullptr;
    return x;
}
template <bool PEER, int K4>
__device__ __forceinline__ void load_item(QRow<K4>& r, const float* row, int l, bool last_ok) {
    if (PEER) r.load_peer(row, l, last_ok); else r.load(row, l, last_ok);
}
template <bool PEER>
__device__ __forceinline__ float load_bias(const float* p) {
    if (!PEER) return __ldg(p);
    float x;
    asm volatile("ld.global.f32 %0, [%1];\n" : "=f"(x) : "l"(p) : "memory");
    return x;
}

template <int K4, int LOSS, bool PEER>
__device__ __forceinline__ void mf_train_fused_q_body(const TrainArgs& a, const PeerArgs& pv) {
    extern __shared__ float sm_scores_all[];   // sampled softmax: [groups per CTA][N1]
    const int lane = threadIdx.x & 31, l = lane & 7;
    const int gid = threadIdx.x >> 3;                                   // group within the CTA
    const int b = blockIdx.x * (kQWarps * 4) + gid;
    const int N1 = a.N1, ld = a.ld, nvec = a.nvec;
    const bool last_ok = l + 8 * (K4 - 1) < nvec;
    // a group past the batch end (or with a bad user index) stays in the loops with everything predicated off: the
    // shuffles below are warp-wide
    int64_t u = 0;
    bool live = b < a.B;
    if (live) {
        u = a.u_idx[b];
        if (bad_index(u, a.n_users)) {
            if (l == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            live = false;
        }
    }
    const int64_t rowoff = (int64_t)(live ? b : 0) * N1;
    const int64_t* __restrict__ irow = a.i_idx + rowoff;
    const bool has_ub = a.Ub != nullptr, has_ib = PEER ? pv.p.Ib[0] != nullptr : a.Ib != nullptr, has_gb = a.Gb != nullptr;
    const uint8_t stamp = PEER ? (uint8_t)(pv.step_dev ? 1 + (int)(*pv.step_dev % 255) : pv.stamp_host) : (uint8_t)0;
    const float ubv = (has_ub && live) ? a.Ub[u] : 0.f, gbv = has_gb ? a.Gb[0] : 0.f;
    const float invf = (float)a.inv_count;

    QRow<K4> ur, gu;
    gu.zero();
    if (live) ur.load(a.Uw + u * ld, l, last_ok); else ur.zero();

    float s0 = 0.f;
    int64_t i0 = 0;
    bool pos_ok = false;
    if (LOSS == HSK_LOSS_BPR) {
        if (live) {
            i0 = irow[0];
            pos_ok = !bad_index(i0, a.n_items);
            if (!pos_ok && l == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        }
        QRow<K4> v0;
        const ItemAt x0 = item_at<PEER>(a, pv, pos_ok ? i0 : 0, ld);
        if (pos_ok) load_item<PEER>(v0, x0.v, l, last_ok); else v0.zero();
        s0 = group_sum(ur.dot(v0));
        if (has_ub) s0 += ubv;
        if (has_ib && pos_ok) s0 += load_bias<PEER>(x0.ib);
        if (has_gb) s0 += gbv;
        live = live && pos_ok;     // a sample whose positive is invalid contributes nothing (as the warp-per-row kernels)
    }
    const int first = (LOSS == HSK_LOSS_BPR) ? 1 : 0;
    float* sm_scores = sm_scores_all + (size_t)gid * N1;
    float ds0 = 0.f, dsum = 0.f, loss_local = 0.f, lse = 0.f;

    // ---- sampled softmax, pass 1: shifted scores of the whole sample -> shared memory, then logsumexp ----
    if (LOSS == HSK_LOSS_SAMPLED_SOFTMAX) {
        for (int j = 0; j < N1; j += kQUnroll) {
            QRow<K4> r[kQUnroll];
            int64_t it[kQUnroll];
            bool ok[kQUnroll];
            float ib[kQUnroll];
#pragma unroll
            for (int q = 0; q < kQUnroll; ++q) {
                ok[q] = live && (j + q < N1);
                it[q] = ok[q] ? irow[j + q] : 0;
                if (ok[q] && bad_index(it[q], a.n_items)) {
                    ok[q] = false;
                    it[q] = 0;
                    if (l == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
                }
            }
#pragma unroll
            for (int q = 0; q < kQUnroll; ++q) {
                const ItemAt x = item_at<PEER>(a, pv, it[q], ld);
                if (ok[q]) load_item<PEER>(r[q], x.v, l, last_ok); else r[q].zero();
                ib[q] = (ok[q] && has_ib) ? load_bias<PEER>(x.ib) : 0.f;
            }
#pragma unroll
            for (int q = 0; q < kQUnroll; ++q) {
                float sj = group_sum(ur.dot(r[q]));
                if (has_ub) sj += ubv;     // sgd_alg.py:173-178 order
                if (has_ib) sj += ib[q];
                if (has_gb) sj += gbv;
                if (l == 0 && j + q < N1) {
                    if (ok[q] && a.scores_out) a.scores_out[rowoff + j + q] = sj;
                    sm_scores[j + q] = ok[q] ? sj + (j + q > 0 ? a.neg_shift : 0.f) : -INFINITY;   // rec_losses.py:131-135
                }
            }
        }
        __syncwarp();
        float mx = -INFINITY;
        for (int j = l; j < N1; j += 8) mx = fmaxf(mx, sm_scores[j]);
        mx = group_max(mx);
        float se = 0.f;
        for (int j = l; j < N1; j += 8) se += expf(sm_scores[j] - mx);
        se = group_sum(se);
        lse = mx + logf(se);
        if (live) loss_local = (lse - sm_scores[0]) * invf;
    }

    // ---- gradients (bpr / bce: scores and gradients in the same pass) ----
    for (int j = first; j < N1; j += kQUnroll) {
        QRow<K4> r[kQUnroll];
        int64_t it[kQUnroll];
        bool ok[kQUnroll];
        float ib[kQUnroll];
        ItemAt at[kQUnroll];
#pragma unroll
        for (int q = 0; q < kQUnroll; ++q) {
            ok[q] = live && (j + q < N1);
            it[q] = ok[q] ? irow[j + q] : 0;
            if (ok[q] && bad_index(it[q], a.n_items)) {
                ok[q] = false;
                it[q] = 0;
                if (LOSS != HSK_LOSS_SAMPLED_SOFTMAX && l == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            }
        }
#pragma unroll
        for (int q = 0; q < kQUnroll; ++q) {
            at[q] = item_at<PEER>(a, pv, it[q], ld);
            if (ok[q]) load_item<PEER>(r[q], at[q].v, l, last_ok); else r[q].zero();
            ib[q] = (LOSS != HSK_LOSS_SAMPLED_SOFTMAX && ok[q] && has_ib) ? load_bias<PEER>(at[q].ib) : 0.f;
        }
#pragma unroll
        for (int q = 0; q < kQUnroll; ++q) {
            float sj = 0.f, dsj;
            if (LOSS != HSK_LOSS_SAMPLED_SOFTMAX) {
                sj = group_sum(ur.dot(r[q]));
                if (has_ub) sj += ubv;
                if (has_ib) sj += ib[q];
                if (has_gb) sj += gbv;
            }
            if (LOSS == HSK_LOSS_BPR) {
                // same arithmetic as hsk_train_tma.cu: one exp serves sigma(x) - 1 and -logsigmoid(x)
                const float x = s0 - sj;
                const float e = expf(-fabsf(x));
                const float rr = __frcp_rn(1.f + e);
                const float dx = ok[q] ? -(x >= 0.f ? e * rr : rr) * invf : 0.f;
                dsj = -dx;
                ds0 += dx;
                if (ok[q]) loss_local += (__logf(1.f + e) - fminf(x, 0.f)) * invf;
            } else if (LOSS == HSK_LOSS_BCE) {
                const float y = (j + q == 0) ? 1.f : 0.f;
                const float e = expf(-fabsf(sj));
                const float rr = __frcp_rn(1.f + e);
                const float sig = sj >= 0.f ? rr : e * rr;
                dsj = ok[q] ? (sig - y) * invf : 0.f;
                if (ok[q]) loss_local += ((1.f - y) * sj + __logf(1.f + e) - fminf(sj, 0.f)) * invf;
            } else {
                dsj = ok[q] ? (expf(sm_scores[j + q] - lse) - (j + q == 0 ? 1.f : 0.f)) * invf : 0.f;
            }
            dsum += dsj;
            gu.axpy(dsj, r[q]);
            if (ok[q]) {
                if (PEER) ur.red_peer(at[q].g, dsj, l, last_ok); else ur.red(at[q].g, dsj, l, last_ok);
                if (l == 0) {
                    if (at[q].gib) { if (PEER) atomicAdd_system(at[q].gib, dsj); else atomicAdd(at[q].gib, dsj); }
                    if (PEER && at[q].st) *at[q].st = stamp;
                    if (LOSS != HSK_LOSS_SAMPLED_SOFTMAX && a.scores_out) a.scores_out[rowoff + j + q] = sj;
                    if (a.dscores_out) a.dscores_out[rowoff + j + q] = dsj;
                }
            }
        }
    }

    // ---- per-sample epilogue: the positive row (bpr), dL/du, bias gradients, loss ----
    if (live) {
        if (LOSS == HSK_LOSS_BPR) {
            QRow<K4> v0;
            const ItemAt x0 = item_at<PEER>(a, pv, i0, ld);
            load_item<PEER>(v0, x0.v, l, last_ok);
            gu.axpy(ds0, v0);
            if (PEER) ur.red_peer(x0.g, ds0, l, last_ok); else ur.red(x0.g, ds0, l, last_ok);
            dsum += ds0;
            if (l == 0) {
                if (x0.gib) { if (PEER) atomicAdd_system(x0.gib, ds0); else atomicAdd(x0.gib, ds0); }
                if (PEER && x0.st) *x0.st = stamp;
                if (a.scores_out) a.scores_out[rowoff] = s0;
                if (a.dscores_out) a.dscores_out[rowoff] = ds0;
            }
        }
        gu.red(a.gU + u * ld, 1.0f, l, last_ok);
        if (l == 0) {
            if (a.gUb) atomicAdd(a.gUb + u, dsum);
            if (a.gGb) atomicAdd(a.gGb, dsum);
        }
    }
    // loss: one double atomic per warp
    double lw = (l == 0) ? (double)loss_local : 0.0;
    lw = warp_sum(lw);
    if (lane == 0 && a.loss_accum && lw != 0.0) atomicAdd(a.loss_accum, lw);
}

template <int K4, int LOSS>
__global__ void __launch_bounds__(kQWarps * 32) mf_train_fused_q_kernel(TrainArgs a) {
    PeerArgs none;     // never read: every use is behind `if (PEER)`
    mf_train_fused_q_body<K4, LOSS, false>(a, none);
}
template <int K4, int LOSS>
__global__ void __launch_bounds__(kQWarps * 32) mf_train_fused_peer_kernel(TrainArgs a, PeerArgs pv) {
    mf_train_fused_q_body<K4, LOSS, true>(a, pv);
}

template <int K4, int LOSS>
__global__ void __launch_bounds__(kQWarps * 32) mf_train_fused_q_pack_kernel(TrainArgs a, PackArgs pk) {
    if (!pack_select_trial(a, pk)) return;
    PeerArgs none;     // never read: every use is behind `if (PEER)`
    mf_train_fused_q_body<K4, LOSS, false>(a, none);
}

template <int LOSS>
static int launch_q_pack(const TrainArgs& a, const PackArgs& pk, int n_active, cudaStream_t s) {
    const int k4 = (a.nvec + 7) / 8;
    const int spc = kQWarps * 4;
    const dim3 grid((a.B + spc - 1) / spc, 1, n_active);
    const size_t smem = (LOSS == HSK_LOSS_SAMPLED_SOFTMAX) ? sizeof(float) * (size_t)spc * a.N1 : 0;
    switch (k4) {
        case 1: mf_train_fused_q_pack_kernel<1, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pk); break;
        case 2: mf_train_fused_q_pack_kernel<2, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pk); break;
        case 3: mf_train_fused_q_pack_kernel<3, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pk); break;
        default: mf_train_fused_q_pack_kernel<4, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pk); break;
    }
    return check_launch("hsk_mf_train_fused_pack(quarter-warp)");
}

int launch_train_fused_q_pack(const TrainArgs& a, const PackArgs& pk, int n_active, int loss_kind, cudaStream_t s) {
    if (loss_kind == HSK_LOSS_BPR) return launch_q_pack<HSK_LOSS_BPR>(a, pk, n_active, s);
    if (loss_kind == HSK_LOSS_BCE) return launch_q_pack<HSK_LOSS_BCE>(a, pk, n_active, s);
    return launch_q_pack<HSK_LOSS_SAMPLED_SOFTMAX>(a, pk, n_active, s);
}

template <int LOSS>
static int launch_q_peer(const TrainArgs& a, const PeerArgs& pv, cudaStream_t s) {
    const int k4 = (a.nvec + 7) / 8;
    const int spc = kQWarps * 4;
    const dim3 grid((a.B + spc - 1) / spc);
    const size_t smem = (LOSS == HSK_LOSS_SAMPLED_SOFTMAX) ? sizeof(float) * (size_t)spc * a.N1 : 0;
    switch (k4) {
        case 1: mf_train_fused_peer_kernel<1, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pv); break;
        case 2: mf_train_fused_peer_kernel<2, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pv); break;
        case 3: mf_train_fused_peer_kernel<3, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pv); break;
        default: mf_train_fused_peer_kernel<4, LOSS><<<grid, kQWarps * 32, smem, s>>>(a, pv); break;
    }
    return check_launch("hsk_mf_train_fused_peer");
}

int launch_train_fused_peer(const TrainArgs& a, const hsk_peer_items& peers, int stamp_host, const int64_t* step_dev, int loss_kind,
                            cudaStream_t s) {
    if (a.nvec > 32) return set_err(HSK_ERR_UNSUPPORTED, "hsk_mf_train_fused_peer: rows of at most 128 floats (ld=%d)", a.ld);
    if (loss_kind == HSK_LOSS_SAMPLED_SOFTMAX && (size_t)a.N1 * kQWarps * 4 * sizeof(float) > 40 * 1024)
        return set_err(HSK_ERR_UNSUPPORTED, "hsk_mf_train_fused_peer: sampled softmax supports at most %d slots per sample",
                       (int)(40 * 1024 / (kQWarps * 4 * sizeof(float))));
    PeerArgs pv;
    pv.p = peers;
    pv.lg = -1;
    for (int b = 0; b < 4; ++b) if ((1 << b) == peers.world) pv.lg = b;
    pv.stamp_host = stamp_host;
    pv.step_dev = step_dev;
    if (loss_kind == HSK_LOSS_BPR) return launch_q_peer<HSK_LOSS_BPR>(a, pv, s);
    if (loss_kind == HSK_LOSS_BCE) return launch_q_peer<HSK_LOSS_BCE>(a, pv, s);
    return launch_q_peer<HSK_LOSS_SAMPLED_SOFTMAX>(a, pv, s);
}

template <int LOSS>
static int launch_q(const TrainArgs& a, cudaStream_t s) {
    const int k4 = (a.nvec + 7) / 8;
    const int spc = kQWarps * 4;   // samples per CTA
    const dim3 grid((a.B + spc - 1) / spc);
    const size_t smem = (LOSS == HSK_LOSS_SAMPLED_SOFTMAX) ? sizeof(float) * (size_t)spc * a.N1 : 0;
    switch (k4) {
        case 1: mf_train_fused_q_kernel<1, LOSS><<<grid, kQWarps * 32, smem, s>>>(a); break;
        case 2: mf_train_fused_q_kernel<2, LOSS><<<grid, kQWarps * 32, smem, s>>>(a); break;
        case 3: mf_train_fused_q_kernel<3, LOSS><<<grid, kQWarps * 32, smem, s>>>(a); break;
        default: mf_train_fused_q_kernel<4, LOSS><<<grid, kQWarps * 32, smem, s>>>(a); break;
    }
    return check_launch("hsk_mf_train_fused(quarter-warp)");
}

// returns 1 (no launch) when the shape is not one this kernel is meant for: rows longer than 128 floats, batches too
// small to fill the GPU with one quarter-warp per sample, softmax samples whose score strip does not fit, or shapes
// where the warp-per-row ring measured faster
bool train_fused_q_fits(int64_t n_samples, int nvec, int N1, int loss_kind, bool force) {
    if (nvec > 32) return false;
    if (!force) {
        if (n_samples < 2048) return false;
        // measured on B200 (B 8192, N 100, tables in L2; scripts/kbench.py trainraw): at d = 128 bpr / bce are bound by L2
        // traffic (reads + REDs) in every layout and the bulk-copy ring is ~10 % ahead (160 vs 176 us); at d = 64 this
        // kernel is 1.9x faster (84 vs 162 us, the ring is bound by its per-row instruction count); sampled softmax
        // (two passes over the rows) is faster here at every d <= 128 (143 vs 165 us at d = 128)
        if (loss_kind != HSK_LOSS_SAMPLED_SOFTMAX && nvec > 24) return false;
    }
    return !(loss_kind == HSK_LOSS_SAMPLED_SOFTMAX && (size_t)N1 * kQWarps * 4 * sizeof(float) > 40 * 1024);
}

int launch_train_fused_q(const TrainArgs& a, int loss_kind, cudaStream_t s) {
    if (!train_fused_q_fits(a.B, a.nvec, a.N1, loss_kind, a.force_q != 0)) return 1;
    if (loss_kind == HSK_LOSS_BPR) return launch_q<HSK_LOSS_BPR>(a, s);
    if (loss_kind == HSK_LOSS_BCE) return launch_q<HSK_LOSS_BCE>(a, s);
    return launch_q<HSK_LOSS_SAMPLED_SOFTMAX>(a, s);
}

}  // namespace hsk
