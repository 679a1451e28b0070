// Device-side routing of the item-sharded training step (SURVEY §8e; replaces what nn.DataParallel does in the
// reference, train/trainer.py:38-40).  World G: item i lives on rank i % G as local row i / G, cap = ceil(n_items / G).
//
// Everything here has FIXED shapes and no host synchronisation, so that the whole sharded step (these kernels, the NCCL
// all-to-alls between them, the fused train kernel and AdamW) can be captured in one CUDA graph:
//
//   hsk_route_items     requester: distinct item ids of the local batch, grouped by owner, numbered in ascending row
//                       order -> req_rows [G, capq] (int32 local rows, -1 padded), compact_idx [n] (row of the compact
//                       table of fetched rows for every batch slot).  No sort: a presence bitmap over the G x cap
//                       owner-major id space + a three-kernel exclusive scan (deterministic numbering).
//   hsk_shard_pack      owner: the rows (and item biases) the peers asked for -> send blocks [G, block_rows, ld]
//   hsk_shard_unpack_add owner: row / bias gradients received back -> added into the dense gradient table, rows stamped
//                       for hsk_adamw_dense_rows
//   hsk_shard_unpack_ordered  the same with the contributions of one row composed in increasing rank order and stored (no
//                       atomics): the owner side of the deterministic 'ordered' exchange
//
// One exchange block per peer is [block_rows, ld] floats: rows [0, capq) are item rows, the floats from row capq on hold
// the capq item biases flat, block_rows = capq + ceil(capq / ld) — so ONE all-to-all moves rows and biases.
#include "hsk_common.cuh"

namespace hsk {

constexpr int kScanBlock = 1024;   // ids per scan block

__global__ void __launch_bounds__(256) route_mark_kernel(const int64_t* __restrict__ idx, int64_t n, int64_t n_items, int G,
                                                         int64_t cap_pad, uint8_t* __restrict__ present, int32_t* status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const int64_t i = idx[e];
        if (bad_index(i, n_items)) {
            if (status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        present[(i % G) * cap_pad + i / G] = 1;
    }
}

// one CTA of 256 threads per scan block of 1024 ids (4 consecutive flag bytes per thread): number of present ids
__global__ void __launch_bounds__(256) route_count_kernel(const uint8_t* __restrict__ present, int32_t* __restrict__ block_count) {
    __shared__ int s_w[8];
    const uint32_t w = reinterpret_cast<const uint32_t*>(present)[(int64_t)blockIdx.x * 256 + threadIdx.x];
    int c = __popc(w & 0x01010101u);
    c = __reduce_add_sync(kFull, c);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += s_w[k];
        block_count[blockIdx.x] = t;
    }
}

// one CTA per owner: exclusive scan of its blocks' counts (any number of blocks, 1024 per round)
__global__ void __launch_bounds__(1024) route_scan_kernel(const int32_t* __restrict__ block_count, int32_t* __restrict__ block_base,
                                                          int blocks_per_owner, int capq, int32_t* __restrict__ req_count,
                                                          int32_t* status) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    const int q = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < blocks_per_owner; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const int c = b < blocks_per_owner ? block_count[q * blocks_per_owner + b] : 0;
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int wv = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(kFull, wv, o);
                if (lane >= o) wv += up;
            }
            s_warp[lane] = wv;   // inclusive over warps
        }
        __syncthreads();
        const int carry = s_carry;
        const int before = carry + (warp > 0 ? s_warp[warp - 1] : 0) + incl - c;
        if (b < blocks_per_owner) block_base[q * blocks_per_owner + b] = before;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int total = s_carry;
        if (total > capq && status) atomicOr(status, HSK_STATUS_CAPACITY);
        req_count[q] = total < capq ? total : capq;
    }
}

// per scan block: slot of every present id = block_base + rank inside the block; req_rows[q, slot] = local row
__global__ void __launch_bounds__(256) route_place_kernel(const uint8_t* __restrict__ present, const int32_t* __restrict__ block_base,
                                                          int blocks_per_owner, int capq, int32_t* __restrict__ slot_of,
                                                          int32_t* __restrict__ req_rows) {
    __shared__ int s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x / blocks_per_owner;
    const int bq = blockIdx.x - q * blocks_per_owner;
    const int64_t j0 = (int64_t)blockIdx.x * kScanBlock + threadIdx.x * 4;   // owner-major index of this thread's first id
    const uint32_t w = reinterpret_cast<const uint32_t*>(present)[(int64_t)blockIdx.x * 256 + threadIdx.x] & 0x01010101u;
    const int c = __popc(w);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int before = block_base[blockIdx.x] + incl - c;
    for (int k = 0; k < warp; ++k) before += s_w[k];
    const int local0 = bq * kScanBlock + threadIdx.x * 4;   // local row of the first id
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        int slot = -1;
        if ((w >> (8 * b)) & 1u) {
            slot = before++;
            if (slot < capq) req_rows[(int64_t)q * capq + slot] = local0 + b; else slot = -1;
        }
        slot_of[j0 + b] = slot;
    }
}

__global__ void __launch_bounds__(256) route_lookup_kernel(const int64_t* __restrict__ idx, int64_t n, int64_t n_items, int G,
                                                           int64_t cap_pad, int64_t block_rows, const int32_t* __restrict__ slot_of,
                                                           int64_t* __restrict__ compact_idx) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const int64_t i = idx[e];
        int64_t out = -1;
        if (!bad_index(i, n_items)) {
            const int q = (int)(i % G);
            const int slot = slot_of[q * cap_pad + i / G];
            if (slot >= 0) out = q * block_rows + slot;
        }
        compact_idx[e] = out;   // -1: bad index or capacity overflow -> the train kernel flags and skips the slot
    }
}

// owner side: one warp per requested row
__global__ void __launch_bounds__(256) shard_pack_kernel(const float* __restrict__ V, const float* __restrict__ Ib, int ld,
                                                         int64_t n_local, const int32_t* __restrict__ rows, int G, int capq,
                                                         int64_t block_rows, float* __restrict__ out, int32_t* status) {
    const int nvec = ld >> 2;
    const int lane = threadIdx.x & 31;
    const int64_t total = (int64_t)G * capq;
    for (int64_t e = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); e < total; e += (int64_t)gridDim.x * 8) {
        const int32_t r = rows[e];
        if (r < 0) continue;
        if (r >= n_local) {
            if (lane == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const int64_t q = e / capq, k = e - q * capq;
        const float4* sp = reinterpret_cast<const float4*>(V + (int64_t)r * ld);
        float4* dp = reinterpret_cast<float4*>(out + (q * block_rows + k) * ld);
        for (int t = lane; t < nvec; t += 32) dp[t] = __ldg(sp + t);
        if (Ib && lane == 0) out[(q * block_rows + capq) * ld + k] = __ldg(Ib + r);
    }
}

__global__ void __launch_bounds__(256) shard_unpack_add_kernel(const float* __restrict__ in, int ld, int64_t n_local,
                                                               const int32_t* __restrict__ rows, int G, int capq, int64_t block_rows,
                                                               float* __restrict__ gV, float* __restrict__ gIb,
                                                               uint8_t* __restrict__ stamps, int stamp_host,
                                                               const int64_t* __restrict__ step_dev, int32_t* status) {
    const int nvec = ld >> 2;
    const int lane = threadIdx.x & 31;
    const int64_t total = (int64_t)G * capq;
    const uint8_t stamp = (uint8_t)(step_dev ? 1 + (int)(*step_dev % 255) : stamp_host);
    for (int64_t e = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); e < total; e += (int64_t)gridDim.x * 8) {
        const int32_t r = rows[e];
        if (r < 0) continue;
        if (r >= n_local) {
            if (lane == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const int64_t q = e / capq, k = e - q * capq;
        const float4* sp = reinterpret_cast<const float4*>(in + (q * block_rows + k) * ld);
        float4* dp = reinterpret_cast<float4*>(gV + (int64_t)r * ld);
        for (int t = lane; t < nvec; t += 32) atomicAdd(dp + t, sp[t]);   // several peers may hold gradients of one row
        if (lane == 0) {
            if (gIb) atomicAdd(gIb + r, in[(q * block_rows + capq) * ld + k]);
            if (stamps) stamps[r] = stamp;
        }
    }
}

// rank-ordered variant (contract in include/hassaku_b200.h, hsk_shard_unpack_ordered): slot of local row r in peer q2's
// request list rows[q2, 0 .. capq) — ascending local rows, then -1 padding — or -1
__device__ __forceinline__ int find_row(const int32_t* __restrict__ list, int capq, int32_t r) {
    int lo = 0, hi = capq;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int32_t v = __ldg(list + mid);
        if (v >= 0 && v < r) lo = mid + 1; else hi = mid;
    }
    return lo < capq && __ldg(list + lo) == r ? lo : -1;
}

__device__ __forceinline__ float4 fadd4_rn(float4 a, float4 b) {
    return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}

// one warp per request entry (q, k); only the entry of the LOWEST rank that fetched the row does the work: it stores that
// rank's contribution, then adds the later ranks' contributions in rank order (their slots found by binary search, 32 ranks
// per round, one per lane) and stamps the row.  Every row has one writer and a fixed summation order: no atomics.
__global__ void __launch_bounds__(256) shard_unpack_ordered_kernel(const float* __restrict__ in, int ld, int64_t n_local,
                                                                   const int32_t* __restrict__ rows, int G, int capq,
                                                                   int64_t block_rows, float* __restrict__ gV,
                                                                   float* __restrict__ gIb, uint8_t* __restrict__ stamps,
                                                                   int stamp_host, const int64_t* __restrict__ step_dev,
                                                                   int32_t* status) {
    __shared__ int s_slot[8][32];
    const int nvec = ld >> 2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t total = (int64_t)G * capq;
    const uint8_t stamp = (uint8_t)(step_dev ? 1 + (int)(*step_dev % 255) : stamp_host);
    for (int64_t e = (int64_t)blockIdx.x * 8 + warp; e < total; e += (int64_t)gridDim.x * 8) {
        const int32_t r = rows[e];
        if (r < 0) continue;
        if (r >= n_local) {
            if (lane == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            continue;
        }
        const int q = (int)(e / capq), k = (int)(e - (int64_t)q * capq);
        bool lower = false;              // a lower rank fetched the row too: its entry is the writer
        for (int b = 0; b < q && !lower; b += 32)
            lower = __any_sync(kFull, b + lane < q && find_row(rows + (int64_t)(b + lane) * capq, capq, r) >= 0);
        if (lower) continue;
        const float4* own = reinterpret_cast<const float4*>(in + ((int64_t)q * block_rows + k) * ld);
        float4* dp = reinterpret_cast<float4*>(gV + (int64_t)r * ld);
        float bias = gIb ? in[((int64_t)q * block_rows + capq) * ld + k] : 0.f;
        int b = q + 1;
        do {                             // ranks b .. b + 31 (the first round also stores this rank's contribution)
            const int q2 = b + lane;
            const int slot = q2 < G ? find_row(rows + (int64_t)q2 * capq, capq, r) : -1;
            unsigned found = __ballot_sync(kFull, slot >= 0);
            s_slot[warp][lane] = slot;
            __syncwarp();
            for (int t = lane; t < nvec; t += 32) {
                float4 acc = b == q + 1 ? own[t] : dp[t];
                for (unsigned m = found; m; m &= m - 1) {
                    const int j = __ffs(m) - 1;
                    const float4* sp = reinterpret_cast<const float4*>(in + ((int64_t)(b + j) * block_rows + s_slot[warp][j]) * ld);
                    acc = fadd4_rn(acc, sp[t]);
                }
                dp[t] = acc;
            }
            if (gIb && lane == 0)
                for (unsigned m = found; m; m &= m - 1) {
                    const int j = __ffs(m) - 1;
                    bias = __fadd_rn(bias, in[((int64_t)(b + j) * block_rows + capq) * ld + s_slot[warp][j]]);
                }
            __syncwarp();
            b += 32;
        } while (b < G);
        if (lane == 0) {
            if (gIb) gIb[r] = bias;
            if (stamps) stamps[r] = stamp;
        }
    }
}

static inline int64_t cap_padded(int64_t n_items, int G) {
    const int64_t cap = (n_items + G - 1) / G;
    return (cap + kScanBlock - 1) / kScanBlock * kScanBlock;
}

}  // namespace hsk

using namespace hsk;

extern "C" int64_t hsk_shard_block_rows(int capq, int ld) { return (int64_t)capq + (capq + ld - 1) / ld; }

extern "C" int64_t hsk_route_scratch_bytes(int64_t n_items, int G) {
    if (n_items < 1 || G < 1) return 0;
    const int64_t cp = cap_padded(n_items, G);
    const int64_t blocks = (int64_t)G * cp / kScanBlock;
    // present (1 B / id) | slot_of (4 B / id) | block_count, block_base (4 B / block each)
    return (int64_t)G * cp * 5 + blocks * 8 + 256;
}

extern "C" int hsk_route_items(const int64_t* i_idx, int64_t n, int64_t n_items, int G, int capq, int ld, int32_t* req_rows,
                               int32_t* req_count, int64_t* compact_idx, void* scratch, int64_t scratch_bytes,
                               int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(req_rows && req_count && scratch && (n == 0 || (i_idx && compact_idx)), "hsk_route_items: null pointer");
    HSK_REQUIRE(n >= 0 && n_items >= 1 && G >= 1 && capq >= 1 && ld >= 4 && ld % 4 == 0, "hsk_route_items: bad sizes");
    HSK_REQUIRE(scratch_bytes >= hsk_route_scratch_bytes(n_items, G), "hsk_route_items: scratch too small");
    HSK_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "hsk_route_items: scratch must be 16-byte aligned");
    const int64_t cp = cap_padded(n_items, G);
    HSK_REQUIRE((int64_t)G * cp < ((int64_t)1 << 31), "hsk_route_items: id space too large");
    const int blocks_per_owner = (int)(cp / kScanBlock);
    const int n_blocks = G * blocks_per_owner;
    uint8_t* present = reinterpret_cast<uint8_t*>(scratch);
    int32_t* slot_of = reinterpret_cast<int32_t*>(present + (int64_t)G * cp);
    int32_t* block_count = slot_of + (int64_t)G * cp;
    int32_t* block_base = block_count + n_blocks;
    cudaStream_t s = as_stream(stream);
    cudaError_t e = cudaMemsetAsync(present, 0, (size_t)G * cp, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(req_rows, 0xFF, sizeof(int32_t) * (size_t)G * capq, s);
    if (e != cudaSuccess) return set_err(HSK_ERR_CUDA, "hsk_route_items: memset: %s", cudaGetErrorString(e));
    const int64_t cap_ctas = (int64_t)sm_count() * 8;
    if (n > 0) {
        const int64_t b = (n + 255) / 256;
        route_mark_kernel<<<(int)(b < cap_ctas ? b : cap_ctas), 256, 0, s>>>(i_idx, n, n_items, G, cp, present, status);
    }
    route_count_kernel<<<n_blocks, 256, 0, s>>>(present, block_count);
    route_scan_kernel<<<G, 1024, 0, s>>>(block_count, block_base, blocks_per_owner, capq, req_count, status);
    route_place_kernel<<<n_blocks, 256, 0, s>>>(present, block_base, blocks_per_owner, capq, slot_of, req_rows);
    if (n > 0) {
        const int64_t b = (n + 255) / 256;
        route_lookup_kernel<<<(int)(b < cap_ctas ? b : cap_ctas), 256, 0, s>>>(i_idx, n, n_items, G, cp, hsk_shard_block_rows(capq, ld),
                                                                               slot_of, compact_idx);
    }
    return check_launch("hsk_route_items");
}

extern "C" int hsk_shard_pack(const float* V, const float* Ib, int ld, int64_t n_local, const int32_t* rows, int G, int capq,
                              float* out, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(V && rows && out, "hsk_shard_pack: null pointer");
    HSK_REQUIRE(ld >= 4 && ld % 4 == 0 && aligned16(V) && aligned16(out) && G >= 1 && capq >= 1 && n_local >= 0, "hsk_shard_pack: bad sizes / alignment");
    const int64_t total = (int64_t)G * capq;
    int64_t blocks = (total + 7) / 8, cap = (int64_t)sm_count() * 16;
    shard_pack_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(V, Ib, ld, n_local, rows, G, capq,
                                                                                         hsk_shard_block_rows(capq, ld), out, status);
    return check_launch("hsk_shard_pack");
}

extern "C" int hsk_shard_unpack_add(const float* in, int ld, int64_t n_local, const int32_t* rows, int G, int capq, float* gV,
                                    float* gIb, uint8_t* stamps, int64_t step, const int64_t* step_dev, int32_t* status,
                                    hsk_stream_t stream) {
    HSK_REQUIRE(in && rows && gV, "hsk_shard_unpack_add: null pointer");
    HSK_REQUIRE(ld >= 4 && ld % 4 == 0 && aligned16(in) && aligned16(gV) && G >= 1 && capq >= 1 && n_local >= 0, "hsk_shard_unpack_add: bad sizes / alignment");
    const int64_t total = (int64_t)G * capq;
    int64_t blocks = (total + 7) / 8, cap = (int64_t)sm_count() * 16;
    shard_unpack_add_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(
        in, ld, n_local, rows, G, capq, hsk_shard_block_rows(capq, ld), gV, gIb, stamps, hsk_row_stamp(step), step_dev, status);
    return check_launch("hsk_shard_unpack_add");
}

extern "C" int hsk_shard_unpack_ordered(const float* in, int ld, int64_t n_local, const int32_t* rows, int G, int capq, float* gV,
                                        float* gIb, uint8_t* stamps, int64_t step, const int64_t* step_dev, int32_t* status,
                                        hsk_stream_t stream) {
    HSK_REQUIRE(in && rows && gV, "hsk_shard_unpack_ordered: null pointer");
    HSK_REQUIRE(ld >= 4 && ld % 4 == 0 && aligned16(in) && aligned16(gV) && G >= 1 && capq >= 1 && n_local >= 0,
                "hsk_shard_unpack_ordered: bad sizes / alignment");
    const int64_t total = (int64_t)G * capq;
    int64_t blocks = (total + 7) / 8, cap = (int64_t)sm_count() * 16;
    shard_unpack_ordered_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, as_stream(stream)>>>(
        in, ld, n_local, rows, G, capq, hsk_shard_block_rows(capq, ld), gV, gIb, stamps, hsk_row_stamp(step), step_dev, status);
    return check_launch("hsk_shard_unpack_ordered");
}
