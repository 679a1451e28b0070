// Argument block shared by the training-step kernels (hsk_train.cu, hsk_train_tma.cu, hsk_train_q.cu).
#pragma once
#include "hsk_common.cuh"

namespace hsk {

constexpr int kWarpsPerCta = 4;

struct TrainArgs {
    const float* __restrict__ Uw;
    const float* __restrict__ Vw;
    const float* __restrict__ Ub;
    const float* __restrict__ Ib;
    const float* __restrict__ Gb;
    float* gU;
    float* gV;
    float* gUb;
    float* gIb;
    float* gGb;
    const int64_t* __restrict__ u_idx;
    const int64_t* __restrict__ i_idx;
    int64_t n_users, n_items;
    int B, N1, ld, nvec;
    int j_per_cta;  // item slots (excluding slot 0) handled by one CTA along gridDim.y
    int loss_kind;
    float neg_shift;
    double inv_count;  // 1/(B*N) bpr, 1/B sampled-softmax, 1/(B*N1) bce
    double* loss_accum;
    float* scores_out;
    float* dscores_out;
    const float* __restrict__ dscores_in;
    int32_t* status;
    int force_q;  // hsk_mf_train_fused_v(variant = quarter-warp): take that kernel whatever the batch size (parity tests)
};

// Trial pack (hsk_mf_train_fused_pack): M models of one shape whose parameter / gradient arenas are the rows of [M, stride]
// allocations.  Kept out of TrainArgs so that the single-model kernels keep their argument layout.
struct PackArgs {
    int64_t stride;           // elements between two trials' arenas (parameters and gradients alike)
    const int32_t* active;    // [gridDim.z] trial indices
    int n_trials;
};

// Points `a` at the tables, gradients and loss accumulator of trial active[blockIdx.z].  False (after flagging the
// status word) when that index is outside [0, n_trials): the CTA then does nothing.
__device__ __forceinline__ bool pack_select_trial(TrainArgs& a, const PackArgs& pk) {
    const int j = pk.active[blockIdx.z];
    if (j < 0 || j >= pk.n_trials) {
        if (threadIdx.x == 0 && a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        return false;
    }
    const int64_t o = (int64_t)j * pk.stride;
    a.Uw += o; a.Vw += o;
    if (a.Ub) a.Ub += o;
    if (a.Ib) a.Ib += o;
    if (a.Gb) a.Gb += o;
    a.gU += o; a.gV += o;
    if (a.gUb) a.gUb += o;
    if (a.gIb) a.gIb += o;
    if (a.gGb) a.gGb += o;
    if (a.loss_accum) a.loss_accum += j;
    return true;
}


// hsk_train_tma.cu: the bulk-copy (TMA) pipelined fused step for bpr / bce; returns HSK_OK or an error code
int launch_train_fused_tma(const TrainArgs& a, int loss_kind, cudaStream_t s);
// hsk_train_q.cu: quarter-warp-per-sample fused step for rows of at most 128 floats; returns 1 (no launch) when the
// shape is outside its range and the caller should use the warp-per-row kernels
int launch_train_fused_q(const TrainArgs& a, int loss_kind, cudaStream_t s);
// hsk_train_q.cu: the shape rule of launch_train_fused_q (n_samples = the samples of all CTAs of the launch)
bool train_fused_q_fits(int64_t n_samples, int nvec, int N1, int loss_kind, bool force);
// hsk_train_q.cu: the quarter-warp kernel over the active trials of a pack (grid z = n_active); no shape rule applied here
int launch_train_fused_q_pack(const TrainArgs& a, const PackArgs& pk, int n_active, int loss_kind, cudaStream_t s);

// hsk_train_q.cu: the same kernel with the item tables sharded over the ranks of a node and mapped into this address
// space (hsk_mf_train_fused_peer): rows gathered from / gradients reduced into the owners' memory over NVLink
int launch_train_fused_peer(const TrainArgs& a, const hsk_peer_items& peers, int stamp_host, const int64_t* step_dev, int loss_kind,
                            cudaStream_t s);

}  // namespace hsk
