// Deterministic mode of the training and evaluation reductions (sm_100a): what runs under
// torch.use_deterministic_algorithms(True).  The default kernels (hsk_train*.cu, hsk_eval.cu) add into shared rows with
// hardware vector reductions whose order depends on timing; the kernels here group the batch by row and give every row
// exactly one writer, so a batch yields the same bits on every run, grid and GPU.
//
//   hsk_mf_scatter_grads_det   backward given dL/dscores: stable radix sort of the batch by item (slots) and by user
//                              (samples), one fixed-order segmented reduction per distinct row, plain stores
//   hsk_mf_train_fused_det     forward + loss + dL/ds per sample (same arithmetic as the fused kernels, dL/ds to scratch,
//                              per-sample fp64 loss), then the scatter above and a fixed-order loss sum
//   hsk_mf_train_fused_det_n   the same with a global normaliser: one rank's share of the sharded 'ordered' step
//   hsk_rec_loss_det           hsk_rec_loss with the per-row losses summed in a fixed order
//   hsk_rank_metrics_sums_det  fixed-order sum of per-user metric rows into the per-group sums
//   hsk_rank_metrics_sums_det_pack  the same for every active trial of a trial pack, batch by batch
//
// ORDER CONTRACT (restated by oracle/det_oracle.py, which reproduces every gradient bit in numpy float32).
//   Slot s = b * N1 + j.  Item side: the n = B * N1 slots are stably sorted by item id, giving positions P = 0 .. n-1
//   (equal ids keep increasing s).  User side: the B samples are stably sorted by user id and every sample expands to its
//   N1 slots, j ascending, giving positions P = 0 .. n-1 (equal ids keep increasing s).  A row's bucket is the run of
//   positions with its id; its entries are in increasing s.
//   Chunks: a bucket is cut at every position P with P % C == 0 (C = 32), i.e. chunk boundaries are the bucket's ends and
//   the multiples of C of the sorted position.  Within a chunk:  acc = +0;  for each entry in order
//       acc = fadd_rn(acc, fmul_rn(ds_s, other_row))      (element-wise; other_row = U[u_b] for items, V[i_s] for users)
//       bias = fadd_rn(bias, ds_s)
//   The row's value is the chunk partials summed in chunk order starting from the first:  r = p0; r = fadd_rn(r, p1); ...
//   and it is STORED (not added) into g: the rows a batch touches are overwritten, the others are not written.
//   Global bias: chunks of CG = 1024 consecutive slots s, summed sequentially from +0 within a chunk, partials summed in
//   order from the first; stored into gGb.
//   The loss: per-sample fp64 terms (as the fused kernels), summed per thread t of 256 over samples t, t+256, ... in order,
//   then a fixed pairwise tree over the 256 partials; loss_accum += that (one plain read-modify-write).
//   Nothing depends on the grid, the SM count or timing: the only atomics left are integer ones (status bits) and
//   shared-memory counters whose results are order-independent.
#include "hsk_train.cuh"

namespace hsk {

constexpr int kDetChunk = 32;      // C of the order contract (== warp width: a chunk is one warp's lane set)
constexpr int kDetGbChunk = 1024;  // CG of the order contract
constexpr int kSortTile = 256;     // elements per radix-sort tile (one per thread)
constexpr int kScanBlock = 1024;   // elements per scan block (one per thread)
static_assert(kDetChunk == 32, "the chunk of the order contract is a warp's lanes");

// ---- scratch layout shared by hsk_det_scratch_bytes and the entry points ----
struct DetPlan {
    int64_t n, n_tiles, n_hist, n_chunks;
    size_t keysA, keysB, valsA, valsB, hist, bsum, part, bpart, gbpart, ds, loss, total;
};

static size_t carve(size_t& off, size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~size_t(255);
    return at;
}

static DetPlan det_plan(int B, int N1, int ld) {
    DetPlan p;
    p.n = (int64_t)B * N1;
    const int64_t n = p.n > 0 ? p.n : 1;
    p.n_tiles = (n + kSortTile - 1) / kSortTile;
    p.n_hist = 256 * p.n_tiles;
    p.n_chunks = (n + kDetChunk - 1) / kDetChunk;
    size_t off = 0;
    p.keysA = carve(off, 4 * (size_t)n);
    p.keysB = carve(off, 4 * (size_t)n);
    p.valsA = carve(off, 4 * (size_t)n);
    p.valsB = carve(off, 4 * (size_t)n);
    p.hist = carve(off, 4 * (size_t)p.n_hist);
    p.bsum = carve(off, 4 * (size_t)((p.n_hist + kScanBlock - 1) / kScanBlock));
    p.part = carve(off, 4 * (size_t)(2 * p.n_chunks) * (size_t)(ld > 0 ? ld : 4));
    p.bpart = carve(off, 4 * (size_t)(2 * p.n_chunks));
    p.gbpart = carve(off, 4 * (size_t)((n + kDetGbChunk - 1) / kDetGbChunk));
    p.ds = carve(off, 4 * (size_t)n);
    p.loss = carve(off, 8 * (size_t)(B > 0 ? B : 1));
    p.total = off;
    return p;
}

// ------------------------------------------------------------------------------------------------
// exclusive scan of an int32 array in place (3 kernels: block sums, scan of the block sums, block scans)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int block_incl_scan_1024(int v, int* s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += up;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(kFull, w, o);
            if (lane >= o) w += up;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    return v + (warp > 0 ? s_warp[warp - 1] : 0);
}

__global__ void __launch_bounds__(kScanBlock) scan_block_sums_kernel(const int32_t* __restrict__ x, int64_t m, int32_t* bsum) {
    __shared__ int s_warp[32];
    const int64_t e = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
    const int incl = block_incl_scan_1024(e < m ? x[e] : 0, s_warp);
    if (threadIdx.x == kScanBlock - 1) bsum[blockIdx.x] = incl;
}

__global__ void __launch_bounds__(kScanBlock) scan_of_sums_kernel(int32_t* bsum, int nb) {
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nb; b0 += kScanBlock) {
        const int b = b0 + threadIdx.x;
        const int c = b < nb ? bsum[b] : 0;
        const int incl = block_incl_scan_1024(c, s_warp);
        const int carry = s_carry;
        if (b < nb) bsum[b] = carry + incl - c;
        __syncthreads();
        if (threadIdx.x == kScanBlock - 1) s_carry = carry + incl;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kScanBlock) scan_apply_kernel(int32_t* x, int64_t m, const int32_t* __restrict__ bsum) {
    __shared__ int s_warp[32];
    const int64_t e = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
    const int v = e < m ? x[e] : 0;
    const int incl = block_incl_scan_1024(v, s_warp);
    if (e < m) x[e] = bsum[blockIdx.x] + incl - v;
}

static int exclusive_scan(int32_t* x, int64_t m, int32_t* bsum, cudaStream_t s) {
    const int nb = (int)((m + kScanBlock - 1) / kScanBlock);
    scan_block_sums_kernel<<<nb, kScanBlock, 0, s>>>(x, m, bsum);
    scan_of_sums_kernel<<<1, kScanBlock, 0, s>>>(bsum, nb);
    scan_apply_kernel<<<nb, kScanBlock, 0, s>>>(x, m, bsum);
    return check_launch("hsk det scan");
}

// ------------------------------------------------------------------------------------------------
// stable LSD radix sort (8-bit digits) of int64 row ids with their element index as payload
// ------------------------------------------------------------------------------------------------
struct SortIn {
    const int64_t* idx;      // first pass: raw ids (validated; a bad id sorts as n_rows), payload = element index
    int64_t n_rows;
    const uint32_t* keys;    // later passes
    const int32_t* vals;
    int32_t* status;
};

__device__ __forceinline__ void sort_load(const SortIn& in, int64_t e, uint32_t& key, int32_t& val) {
    if (in.idx) {
        const int64_t v = in.idx[e];
        if (bad_index(v, in.n_rows)) {
            key = (uint32_t)in.n_rows;
            if (in.status) atomicOr(in.status, HSK_STATUS_BAD_INDEX);
        } else {
            key = (uint32_t)v;
        }
        val = (int32_t)e;
    } else {
        key = in.keys[e];
        val = in.vals[e];
    }
}

// rank of this thread's element among the preceding elements of the tile with the same digit (digit < 0: no element);
// returns in `count` the tile's number of elements whose digit is threadIdx.x
__device__ __forceinline__ int tile_rank(int digit, int (*wcnt)[256], int& count) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int w = 0; w < kSortTile / 32; ++w) wcnt[w][threadIdx.x] = 0;
    __syncthreads();
    const unsigned m = __match_any_sync(kFull, digit);
    const int lrank = __popc(m & ((1u << lane) - 1u));
    if (digit >= 0 && lrank == 0) wcnt[warp][digit] = __popc(m);
    __syncthreads();
    int run = 0;
#pragma unroll
    for (int w = 0; w < kSortTile / 32; ++w) {
        const int c = wcnt[w][threadIdx.x];
        wcnt[w][threadIdx.x] = run;
        run += c;
    }
    count = run;
    __syncthreads();
    return digit >= 0 ? wcnt[warp][digit] + lrank : 0;
}

__global__ void __launch_bounds__(kSortTile) sort_hist_kernel(SortIn in, int64_t n, int shift, int64_t n_tiles, int32_t* hist) {
    __shared__ int wcnt[kSortTile / 32][256];
    const int64_t e = (int64_t)blockIdx.x * kSortTile + threadIdx.x;
    int digit = -1;
    if (e < n) {
        uint32_t key; int32_t val;
        sort_load(in, e, key, val);
        digit = (int)((key >> shift) & 255u);
    }
    int count;
    tile_rank(digit, wcnt, count);
    hist[(int64_t)threadIdx.x * n_tiles + blockIdx.x] = count;
}

__global__ void __launch_bounds__(kSortTile) sort_scatter_kernel(SortIn in, int64_t n, int shift, int64_t n_tiles,
                                                                 const int32_t* __restrict__ base, uint32_t* keys_out,
                                                                 int32_t* vals_out) {
    __shared__ int wcnt[kSortTile / 32][256];
    const int64_t e = (int64_t)blockIdx.x * kSortTile + threadIdx.x;
    int digit = -1;
    uint32_t key = 0; int32_t val = 0;
    if (e < n) {
        in.status = nullptr;   // reported by the histogram pass
        sort_load(in, e, key, val);
        digit = (int)((key >> shift) & 255u);
    }
    int count;
    const int rank = tile_rank(digit, wcnt, count);
    if (digit >= 0) {
        const int64_t pos = base[(int64_t)digit * n_tiles + blockIdx.x] + rank;
        keys_out[pos] = key;
        vals_out[pos] = val;
    }
}

// sorts ids idx[0 .. n) (< n_rows, else keyed n_rows); the result is left in (*keys, *vals)
static int radix_sort(const int64_t* idx, int64_t n, int64_t n_rows, char* base, const DetPlan& p, int32_t* status,
                      const uint32_t** keys, const int32_t** vals, cudaStream_t s) {
    uint32_t* kbuf[2] = {reinterpret_cast<uint32_t*>(base + p.keysA), reinterpret_cast<uint32_t*>(base + p.keysB)};
    int32_t* vbuf[2] = {reinterpret_cast<int32_t*>(base + p.valsA), reinterpret_cast<int32_t*>(base + p.valsB)};
    int32_t* hist = reinterpret_cast<int32_t*>(base + p.hist);
    int32_t* bsum = reinterpret_cast<int32_t*>(base + p.bsum);
    const int bits = 64 - __builtin_clzll((unsigned long long)n_rows);   // keys <= n_rows
    const int passes = bits > 8 ? (bits + 7) / 8 : 1;
    const int64_t n_tiles = (n + kSortTile - 1) / kSortTile;
    SortIn in{idx, n_rows, nullptr, nullptr, status};
    int cur = 0;
    for (int pass = 0; pass < passes; ++pass) {
        const int shift = 8 * pass;
        sort_hist_kernel<<<(unsigned)n_tiles, kSortTile, 0, s>>>(in, n, shift, n_tiles, hist);
        int rc = exclusive_scan(hist, 256 * n_tiles, bsum, s);
        if (rc) return rc;
        sort_scatter_kernel<<<(unsigned)n_tiles, kSortTile, 0, s>>>(in, n, shift, n_tiles, hist, kbuf[cur], vbuf[cur]);
        in = SortIn{nullptr, n_rows, kbuf[cur], vbuf[cur], nullptr};
        cur ^= 1;
    }
    *keys = kbuf[cur ^ 1];
    *vals = vbuf[cur ^ 1];
    return check_launch("hsk det radix sort");
}

// ------------------------------------------------------------------------------------------------
// segmented reductions over the sorted positions (order contract above)
// ------------------------------------------------------------------------------------------------
struct SegArgs {
    const uint32_t* skey;                // sorted ids: [n] (items) or [B] (users)
    const int32_t* sval;                 // their slot (items) or sample (users)
    const float* __restrict__ other;     // U (items side) or V (users side)
    int64_t n_other;
    const int64_t* __restrict__ u_idx;
    const int64_t* __restrict__ i_idx;
    const float* __restrict__ ds;        // dL/dscores [B, N1]
    int64_t n;                           // B * N1 positions
    int N1, ld, nvec;
    int64_t n_rows;                      // ids >= n_rows (the bad-index key) are skipped
    float* g;                            // gV / gU
    float* gb;                           // gIb / gUb (nullable)
    float* part;                         // [2 * n_chunks, ld]
    float* bpart;                        // [2 * n_chunks]
};

template <bool USER>
__device__ __forceinline__ uint32_t key_at(const SegArgs& a, int64_t P) { return a.skey[USER ? P / a.N1 : P]; }
template <bool USER>
__device__ __forceinline__ int64_t slot_at(const SegArgs& a, int64_t P) {
    return USER ? (int64_t)a.sval[P / a.N1] * a.N1 + P % a.N1 : (int64_t)a.sval[P];
}

template <int NV>
__device__ __forceinline__ void axpy_rn(Row<NV>& acc, float d, const Row<NV>& x) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        acc.v[k].x = __fadd_rn(acc.v[k].x, __fmul_rn(d, x.v[k].x));
        acc.v[k].y = __fadd_rn(acc.v[k].y, __fmul_rn(d, x.v[k].y));
        acc.v[k].z = __fadd_rn(acc.v[k].z, __fmul_rn(d, x.v[k].z));
        acc.v[k].w = __fadd_rn(acc.v[k].w, __fmul_rn(d, x.v[k].w));
    }
}
template <int NV>
__device__ __forceinline__ void add_rn(Row<NV>& acc, const Row<NV>& x) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        acc.v[k].x = __fadd_rn(acc.v[k].x, x.v[k].x);
        acc.v[k].y = __fadd_rn(acc.v[k].y, x.v[k].y);
        acc.v[k].z = __fadd_rn(acc.v[k].z, x.v[k].z);
        acc.v[k].w = __fadd_rn(acc.v[k].w, x.v[k].w);
    }
}
template <int NV>
__device__ __forceinline__ void store_row(const Row<NV>& r, float* dst, int nvec, int lane) {
    float4* p = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const int idx = lane + 32 * k;
        if (idx < nvec) p[idx] = r.v[k];
    }
}

// one warp per chunk head: the chunk's entries in order; a one-chunk bucket stores its row, else the chunk's partial
template <int NV, bool USER>
__global__ void __launch_bounds__(256) det_chunk_kernel(SegArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t P = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (P >= a.n) return;
    const uint32_t key = key_at<USER>(a, P);
    const bool starts = P == 0 || key_at<USER>(a, P - 1) != key;
    if ((!starts && P % kDetChunk != 0) || key >= a.n_rows) return;
    const int64_t end = min(a.n, (P / kDetChunk + 1) * kDetChunk);
    const int64_t q = P + lane;
    const bool in = q < end && key_at<USER>(a, q) == key;
    const int L = __popc(__ballot_sync(kFull, in));   // the bucket is contiguous: the lanes in it are a prefix
    int64_t o = -1;
    float d = 0.f;
    if (in) {
        const int64_t s = slot_at<USER>(a, q);
        o = USER ? a.i_idx[s] : a.u_idx[s / a.N1];
        if (bad_index(o, a.n_other)) o = -1;
        d = a.ds[s];
    }
    Row<NV> acc;
    acc.zero();
    float bacc = 0.f;
#pragma unroll 2
    for (int k = 0; k < L; ++k) {
        const int64_t ok = __shfl_sync(kFull, o, k);
        const float dk = __shfl_sync(kFull, d, k);
        if (ok < 0) continue;
        Row<NV> r;
        r.load(a.other + ok * a.ld, a.nvec, lane);
        axpy_rn(acc, dk, r);
        bacc = __fadd_rn(bacc, dk);
    }
    const bool continues = P + L == end && end < a.n && key_at<USER>(a, end) == key;
    if (starts && !continues) {
        store_row(acc, a.g + (int64_t)key * a.ld, a.nvec, lane);
        if (lane == 0 && a.gb) a.gb[key] = bacc;
    } else {
        const int64_t slot = 2 * (P / kDetChunk) + (P % kDetChunk != 0 ? 1 : 0);
        store_row(acc, a.part + slot * a.ld, a.nvec, lane);
        if (lane == 0) a.bpart[slot] = bacc;
    }
}

// one warp per aligned block of C positions: the bucket that starts in it and crosses its end sums its chunk partials
template <int NV, bool USER>
__global__ void __launch_bounds__(256) det_combine_kernel(SegArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int64_t lo = m * kDetChunk;
    if (lo >= a.n) return;
    const int64_t e = min(a.n, lo + kDetChunk) - 1;
    if (e + 1 >= a.n) return;
    const uint32_t key = key_at<USER>(a, e);
    if (key >= a.n_rows || key_at<USER>(a, e + 1) != key) return;
    if (m > 0 && key_at<USER>(a, lo - 1) == key) return;   // started in an earlier block, which owns it
    const int64_t x = lo + lane;
    const unsigned bal = __ballot_sync(kFull, x <= e && key_at<USER>(a, x) == key);
    const int64_t p0 = lo + __ffs(bal) - 1;
    const int64_t slot0 = 2 * m + (p0 != lo ? 1 : 0);
    Row<NV> acc;
    acc.load(a.part + slot0 * a.ld, a.nvec, lane);
    float bacc = a.bpart[slot0];
    for (int64_t m2 = m + 1; m2 * kDetChunk < a.n && key_at<USER>(a, m2 * kDetChunk) == key; ++m2) {
        Row<NV> r;
        r.load(a.part + 2 * m2 * a.ld, a.nvec, lane);
        add_rn(acc, r);
        bacc = __fadd_rn(bacc, a.bpart[2 * m2]);
    }
    store_row(acc, a.g + (int64_t)key * a.ld, a.nvec, lane);
    if (lane == 0 && a.gb) a.gb[key] = bacc;
}

// global bias: chunk partials of CG consecutive slots, then their ordered sum (one thread)
__global__ void __launch_bounds__(128) gb_chunk_kernel(const float* __restrict__ ds, int64_t n, float* gbpart) {
    const int64_t c = (int64_t)blockIdx.x * 128 + threadIdx.x;
    const int64_t s0 = c * kDetGbChunk;
    if (s0 >= n) return;
    const int64_t s1 = min(n, s0 + kDetGbChunk);
    float acc = 0.f;
    for (int64_t s = s0; s < s1; ++s) acc = __fadd_rn(acc, ds[s]);
    gbpart[c] = acc;
}
__global__ void gb_final_kernel(const float* __restrict__ gbpart, int64_t n_chunks, float* gGb) {
    float acc = gbpart[0];
    for (int64_t c = 1; c < n_chunks; ++c) acc = __fadd_rn(acc, gbpart[c]);
    gGb[0] = acc;
}

// ------------------------------------------------------------------------------------------------
// loss + dL/ds of one sample row (one warp): the arithmetic of rec_loss_kernel (hsk_train.cu); returns the row's loss
// on every lane.  ds2 (nullable) receives a copy of ds.  shifted may alias s (sampled-softmax in-place shift).
// ------------------------------------------------------------------------------------------------
__device__ double loss_row(const float* s, const double* lab, int N1, int kind, float shift, float gscale, int B, float* ds,
                           float* ds2, float* shifted) {
    const int lane = threadIdx.x & 31;
    double loss = 0.0;
    if (kind == HSK_LOSS_BPR) {
        const double inv = 1.0 / ((double)B * (double)(N1 - 1));
        const float s0 = s[0];
        const double y = lab ? lab[0] : 1.0;
        float ds0 = 0.f;
        for (int j = 1 + lane; j < N1; j += 32) {
            const float x = s0 - s[j];
            loss += ((1.0 - y) * (double)x - (double)log_sigmoid_f(x)) * inv;
            const float dx = (float)(((double)sigmoid_f(x) - y) * inv) * gscale;
            ds[j] = -dx;
            if (ds2) ds2[j] = -dx;
            ds0 += dx;
        }
        ds0 = warp_sum(ds0);
        if (lane == 0) {
            ds[0] = ds0;
            if (ds2) ds2[0] = ds0;
        }
    } else if (kind == HSK_LOSS_SAMPLED_SOFTMAX) {
        float mx = -INFINITY;
        for (int j = lane; j < N1; j += 32) mx = fmaxf(mx, s[j] + (j > 0 ? shift : 0.f));
        mx = warp_max(mx);
        float se = 0.f;
        for (int j = lane; j < N1; j += 32) se += expf(s[j] + (j > 0 ? shift : 0.f) - mx);
        se = warp_sum(se);
        const float lse = mx + logf(se);
        const float s0 = s[0];
        __syncwarp();
        const float invB = 1.f / (float)B;
        for (int j = lane; j < N1; j += 32) {
            const float x = s[j] + (j > 0 ? shift : 0.f);
            const float d = (expf(x - lse) - (j == 0 ? 1.f : 0.f)) * invB * gscale;
            ds[j] = d;
            if (ds2) ds2[j] = d;
            if (shifted) shifted[j] = x;
        }
        if (lane == 0) loss = (double)(lse - s0) / (double)B;
    } else {
        const double inv = 1.0 / ((double)B * (double)N1);
        for (int j = lane; j < N1; j += 32) {
            const float x = s[j];
            const double y = lab ? lab[j] : (j == 0 ? 1.0 : 0.0);
            loss += ((1.0 - y) * (double)x - (double)log_sigmoid_f(x)) * inv;
            const float d = (float)(((double)sigmoid_f(x) - y) * inv) * gscale;
            ds[j] = d;
            if (ds2) ds2[j] = d;
        }
    }
    return warp_sum(loss);
}

// fused forward: one CTA of 4 warps per sample, scores to shared memory, then warp 0 produces the loss row and dL/ds.
// A sample with an out-of-range user or item index is skipped (dL/ds 0, loss 0) and reported in status.
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32) det_forward_kernel(TrainArgs a, float* __restrict__ ds, double* __restrict__ loss_rows) {
    extern __shared__ float sm_s[];
    __shared__ int sm_bad;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x;
    const int64_t u = a.u_idx[b];
    const int64_t* irow = a.i_idx + (int64_t)b * a.N1;
    const int64_t rowoff = (int64_t)b * a.N1;
    if (threadIdx.x == 0) sm_bad = bad_index(u, a.n_users) ? 1 : 0;
    __syncthreads();
    if (!sm_bad) {
        Row<NV> ur;
        ur.load(a.Uw + u * a.ld, a.nvec, lane);
        const float bias_u = a.Ub ? a.Ub[u] : 0.f;
        const float gb = a.Gb ? a.Gb[0] : 0.f;
        for (int j = warp; j < a.N1; j += kWarpsPerCta) {
            const int64_t it = irow[j];
            if (bad_index(it, a.n_items)) {
                if (lane == 0) sm_bad = 1;
                continue;
            }
            Row<NV> vr;
            vr.load(a.Vw + it * a.ld, a.nvec, lane);
            float sj = warp_sum(ur.dot_partial(vr));
            if (a.Ub) sj += bias_u;
            if (a.Ib) sj += a.Ib[it];
            if (a.Gb) sj += gb;
            if (lane == 0) sm_s[j] = sj;
        }
    }
    __syncthreads();
    if (warp != 0) return;
    if (sm_bad) {
        for (int j = lane; j < a.N1; j += 32) {
            ds[rowoff + j] = 0.f;
            if (a.dscores_out) a.dscores_out[rowoff + j] = 0.f;
        }
        if (lane == 0) {
            loss_rows[b] = 0.0;
            if (a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
        }
        return;
    }
    if (a.scores_out)
        for (int j = lane; j < a.N1; j += 32) a.scores_out[rowoff + j] = sm_s[j];
    const double l = loss_row(sm_s, nullptr, a.N1, a.loss_kind, a.neg_shift, 1.f, a.B, ds + rowoff,
                              a.dscores_out ? a.dscores_out + rowoff : nullptr, nullptr);
    if (lane == 0) loss_rows[b] = l;
}

// hsk_rec_loss_det: one warp per row of a score matrix
__global__ void __launch_bounds__(256) det_rec_loss_kernel(const float* scores, const double* __restrict__ labels, int B, int N1,
                                                           int kind, float shift, float gscale, float* dscores, float* shifted_out,
                                                           double* __restrict__ loss_rows) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const int64_t off = (int64_t)b * N1;
    const double l = loss_row(scores + off, labels ? labels + off : nullptr, N1, kind, shift, gscale, B, dscores + off, nullptr,
                              shifted_out ? shifted_out + off : nullptr);
    if ((threadIdx.x & 31) == 0) loss_rows[b] = l;
}

// loss_accum += the fixed-order sum of the per-sample losses (one CTA of 256 threads)
__global__ void __launch_bounds__(256) det_loss_sum_kernel(const double* __restrict__ loss_rows, int B, double* loss_accum) {
    __shared__ double sm[256];
    double acc = 0.0;
    for (int b = threadIdx.x; b < B; b += 256) acc = __dadd_rn(acc, loss_rows[b]);
    sm[threadIdx.x] = acc;
    __syncthreads();
#pragma unroll
    for (int w = 128; w > 0; w >>= 1) {
        if (threadIdx.x < w) sm[threadIdx.x] = __dadd_rn(sm[threadIdx.x], sm[threadIdx.x + w]);
        __syncthreads();
    }
    if (threadIdx.x == 0) loss_accum[0] = __dadd_rn(loss_accum[0], sm[0]);
}

// sums[g] += the fixed-order sum over the batch's users of group g - 1 (g = 0: all users) of per_user [Be, n_cells]
__global__ void __launch_bounds__(256) det_metric_sums_kernel(const float* __restrict__ per_user, int Be, int n_cells,
                                                              const int64_t* __restrict__ u_idx, const int32_t* __restrict__ group,
                                                              int n_groups, double* sums) {
#include "hsk_det_metric_sums_body.inc"
}

// trial pack (hsk_rank_metrics_sums_det_pack): gridDim.y walks the active trials; per trial the rows are cut into batches of
// `batch` and each batch is added by the body above, in order, into the trial's sums
__global__ void __launch_bounds__(256) det_metric_sums_pack_kernel(const float* __restrict__ per_user_all, int Be_all, int batch,
                                                                   int n_cells, const int64_t* __restrict__ u_all,
                                                                   const int32_t* __restrict__ group, int n_groups, int groups,
                                                                   const int32_t* __restrict__ active, int n_trials,
                                                                   double* sums_all, int32_t* status) {
    const int jt = active[blockIdx.y];
    if (jt < 0 || jt >= n_trials) {
        if (threadIdx.x == 0 && status) atomicOr(status, HSK_STATUS_BAD_INDEX);
        return;
    }
    double* sums = sums_all + (int64_t)jt * (1 + groups) * n_cells;
    for (int b0 = 0; b0 < Be_all; b0 += batch) {
        const float* __restrict__ per_user = per_user_all + ((int64_t)blockIdx.y * Be_all + b0) * n_cells;
        const int Be = min(batch, Be_all - b0);
        const int64_t* __restrict__ u_idx = u_all + b0;
        {
#include "hsk_det_metric_sums_body.inc"
        }
    }
}

// ---- host: the scatter of one batch given dL/ds (device) ----
template <int NV>
static int det_scatter_nv(const TrainArgs& a, const float* ds, char* base, const DetPlan& p, cudaStream_t s) {
    const int64_t n = p.n;
    SegArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.u_idx = a.u_idx; sa.i_idx = a.i_idx; sa.ds = ds; sa.n = n;
    sa.N1 = a.N1; sa.ld = a.ld; sa.nvec = a.nvec;
    sa.part = reinterpret_cast<float*>(base + p.part);
    sa.bpart = reinterpret_cast<float*>(base + p.bpart);
    const unsigned grid_pos = (unsigned)((n + 7) / 8), grid_blk = (unsigned)((p.n_chunks + 7) / 8);
    // item rows
    int rc = radix_sort(a.i_idx, n, a.n_items, base, p, a.status, &sa.skey, &sa.sval, s);
    if (rc) return rc;
    sa.other = a.Uw; sa.n_other = a.n_users; sa.n_rows = a.n_items; sa.g = a.gV; sa.gb = a.gIb;
    det_chunk_kernel<NV, false><<<grid_pos, 256, 0, s>>>(sa);
    det_combine_kernel<NV, false><<<grid_blk, 256, 0, s>>>(sa);
    // user rows (the sort buffers and partials are reused: same stream)
    rc = radix_sort(a.u_idx, a.B, a.n_users, base, p, a.status, &sa.skey, &sa.sval, s);
    if (rc) return rc;
    sa.other = a.Vw; sa.n_other = a.n_items; sa.n_rows = a.n_users; sa.g = a.gU; sa.gb = a.gUb;
    det_chunk_kernel<NV, true><<<grid_pos, 256, 0, s>>>(sa);
    det_combine_kernel<NV, true><<<grid_blk, 256, 0, s>>>(sa);
    if (a.gGb) {
        float* gbpart = reinterpret_cast<float*>(base + p.gbpart);
        const int64_t nc = (n + kDetGbChunk - 1) / kDetGbChunk;
        gb_chunk_kernel<<<(unsigned)((nc + 127) / 128), 128, 0, s>>>(ds, n, gbpart);
        gb_final_kernel<<<1, 1, 0, s>>>(gbpart, nc, a.gGb);
    }
    return check_launch("hsk det scatter");
}

static int det_scatter(const TrainArgs& a, const float* ds, char* base, const DetPlan& p, cudaStream_t s) {
    const int nv = (a.nvec + 31) / 32;
    HSK_DISPATCH_NV(nv, return det_scatter_nv<NV>(a, ds, base, p, s));
    return HSK_OK;
}

static int det_args(TrainArgs& a, const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                    int B, int N1, void* scratch, int64_t scratch_bytes, DetPlan& p, const char* who) {
    HSK_REQUIRE(t && t->Uw && t->Vw && g && g->Uw && g->Vw && u_idx && i_idx, "%s: null pointer", who);
    HSK_REQUIRE(B >= 0 && N1 >= 1 && (int64_t)B * N1 < 0x7FFFFFFFll, "%s: need B >= 0, N1 >= 1, B * N1 < 2^31", who);
    HSK_REQUIRE(t->d >= 1 && t->ld >= t->d && (t->ld % 4) == 0, "%s: need 1 <= d <= ld and ld %% 4 == 0", who);
    HSK_REQUIRE(t->n_users >= 1 && t->n_items >= 1 && t->n_users < 0x7FFFFFFFll && t->n_items < 0x7FFFFFFFll,
                "%s: table row counts must be in [1, 2^31)", who);
    HSK_REQUIRE(g->ld == t->ld && g->d == t->d && g->n_users == t->n_users && g->n_items == t->n_items,
                "%s: gradient tables must have the layout of the parameter tables", who);
    HSK_REQUIRE(aligned16(t->Uw) && aligned16(t->Vw) && aligned16(g->Uw) && aligned16(g->Vw), "%s: tables must be 16-byte aligned", who);
    HSK_REQUIRE((!t->Ub || g->Ub) && (!t->Ib || g->Ib) && (!t->Gb || g->Gb), "%s: missing bias gradient buffer", who);
    p = det_plan(B, N1, t->ld);
    HSK_REQUIRE(scratch && aligned16(scratch) && scratch_bytes >= (int64_t)p.total, "%s: scratch too small (%lld < %lld bytes)", who,
                (long long)scratch_bytes, (long long)p.total);
    memset(&a, 0, sizeof(a));
    a.Uw = t->Uw; a.Vw = t->Vw; a.Ub = t->Ub; a.Ib = t->Ib; a.Gb = t->Gb;
    a.gU = g->Uw; a.gV = g->Vw; a.gUb = t->Ub ? g->Ub : nullptr; a.gIb = t->Ib ? g->Ib : nullptr; a.gGb = t->Gb ? g->Gb : nullptr;
    a.n_users = t->n_users; a.n_items = t->n_items;
    a.B = B; a.N1 = N1; a.ld = t->ld; a.nvec = t->ld / 4;
    a.u_idx = u_idx; a.i_idx = i_idx;
    return HSK_OK;
}

}  // namespace hsk

using namespace hsk;

extern "C" int64_t hsk_det_scratch_bytes(int B, int N1, int ld) { return (int64_t)det_plan(B, N1, ld).total; }

extern "C" int hsk_mf_scatter_grads_det(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                        const float* dscores, int B, int N1, void* scratch, int64_t scratch_bytes, int32_t* status,
                                        hsk_stream_t stream) {
    TrainArgs a;
    DetPlan p;
    int rc = det_args(a, t, g, u_idx, i_idx, B, N1, scratch, scratch_bytes, p, "hsk_mf_scatter_grads_det");
    if (rc) return rc;
    HSK_REQUIRE(dscores, "hsk_mf_scatter_grads_det: dscores is null");
    if (B == 0) return HSK_OK;
    a.status = status;
    return det_scatter(a, dscores, static_cast<char*>(scratch), p, as_stream(stream));
}

// B_global: the loss / gradient normaliser (the whole step's batch when this is one rank's share of it); the forward,
// sorts, scatter and loss sum run on the local B
static int train_fused_det(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx, int B,
                           int N1, int64_t B_global, int loss_kind, float neg_shift, double* loss_accum, float* scores_out,
                           float* dscores_out, void* scratch, int64_t scratch_bytes, int32_t* status, hsk_stream_t stream,
                           const char* who) {
    TrainArgs a;
    DetPlan p;
    int rc = det_args(a, t, g, u_idx, i_idx, B, N1, scratch, scratch_bytes, p, who);
    if (rc) return rc;
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "%s: unknown loss kind %d", who, loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "%s: bpr needs at least one negative", who);
    HSK_REQUIRE(N1 <= 10240, "%s: at most 10240 slots per sample", who);
    HSK_REQUIRE(B_global >= B && B_global <= 0x7FFFFFFFll, "%s: need B <= B_global < 2^31", who);
    if (B == 0) return HSK_OK;
    a.status = status; a.loss_kind = loss_kind; a.neg_shift = neg_shift;
    a.scores_out = scores_out; a.dscores_out = dscores_out;
    char* base = static_cast<char*>(scratch);
    float* ds = reinterpret_cast<float*>(base + p.ds);
    double* loss_rows = reinterpret_cast<double*>(base + p.loss);
    cudaStream_t s = as_stream(stream);
    const int nv = (a.nvec + 31) / 32;
    const size_t smem = sizeof(float) * (size_t)N1;
    // det_forward_kernel reads a.B only as loss_row's normaliser (the sample is blockIdx.x): the grid stays the local B
    TrainArgs fa = a;
    fa.B = (int)B_global;
    HSK_DISPATCH_NV(nv, (det_forward_kernel<NV><<<B, kWarpsPerCta * 32, smem, s>>>(fa, ds, loss_rows)));
    rc = check_launch(who);
    if (rc) return rc;
    if (loss_accum) det_loss_sum_kernel<<<1, 256, 0, s>>>(loss_rows, B, loss_accum);
    return det_scatter(a, ds, base, p, s);
}

extern "C" int hsk_mf_train_fused_det(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                      int B, int N1, int loss_kind, float neg_shift, double* loss_accum, float* scores_out,
                                      float* dscores_out, void* scratch, int64_t scratch_bytes, int32_t* status,
                                      hsk_stream_t stream) {
    return train_fused_det(t, g, u_idx, i_idx, B, N1, B, loss_kind, neg_shift, loss_accum, scores_out, dscores_out, scratch,
                           scratch_bytes, status, stream, "hsk_mf_train_fused_det");
}

extern "C" int hsk_mf_train_fused_det_n(const hsk_mf_tables* t, const hsk_mf_tables* g, const int64_t* u_idx, const int64_t* i_idx,
                                        int B, int N1, int64_t B_global, int loss_kind, float neg_shift, double* loss_accum,
                                        float* scores_out, float* dscores_out, void* scratch, int64_t scratch_bytes,
                                        int32_t* status, hsk_stream_t stream) {
    static const int64_t kNoIndex = 0;
    if (B == 0) {     // a rank without samples in this step: nothing is launched, its (empty) index arrays may be null
        if (!u_idx) u_idx = &kNoIndex;
        if (!i_idx) i_idx = &kNoIndex;
    }
    return train_fused_det(t, g, u_idx, i_idx, B, N1, B_global, loss_kind, neg_shift, loss_accum, scores_out, dscores_out,
                           scratch, scratch_bytes, status, stream, "hsk_mf_train_fused_det_n");
}

extern "C" int hsk_rec_loss_det(const float* scores, const double* labels, int B, int N1, int loss_kind, float neg_shift,
                                float grad_scale, double* loss_accum, float* dscores, float* shifted_out, void* scratch,
                                int64_t scratch_bytes, hsk_stream_t stream) {
    HSK_REQUIRE(scores && loss_accum && dscores, "hsk_rec_loss_det: scores, loss_accum and dscores are required");
    HSK_REQUIRE(dscores != scores, "hsk_rec_loss_det: dscores may not alias scores");
    HSK_REQUIRE(B >= 0 && N1 >= 1, "hsk_rec_loss_det: need B >= 0, N1 >= 1");
    HSK_REQUIRE(loss_kind >= 0 && loss_kind <= 2, "hsk_rec_loss_det: unknown loss kind %d", loss_kind);
    HSK_REQUIRE(loss_kind != HSK_LOSS_BPR || N1 >= 2, "hsk_rec_loss_det: bpr needs at least one negative");
    HSK_REQUIRE(scratch && aligned16(scratch) && scratch_bytes >= 8 * (int64_t)B, "hsk_rec_loss_det: scratch needs 8 * B bytes");
    if (B == 0) return HSK_OK;
    double* loss_rows = static_cast<double*>(scratch);
    cudaStream_t s = as_stream(stream);
    det_rec_loss_kernel<<<(B + 7) / 8, 256, 0, s>>>(scores, labels, B, N1, loss_kind, neg_shift, grad_scale, dscores, shifted_out,
                                                    loss_rows);
    det_loss_sum_kernel<<<1, 256, 0, s>>>(loss_rows, B, loss_accum);
    return check_launch("hsk_rec_loss_det");
}

extern "C" int hsk_rank_metrics_sums_det(const float* per_user, int Be, int n_ks, const int64_t* u_idx, const int32_t* user_group,
                                         int n_groups, double* sums, hsk_stream_t stream) {
    HSK_REQUIRE(per_user && u_idx && sums, "hsk_rank_metrics_sums_det: null pointer");
    HSK_REQUIRE(n_ks >= 1 && n_ks <= 8 && n_groups >= 0 && Be >= 0, "hsk_rank_metrics_sums_det: need 1 <= n_ks <= 8");
    if (Be == 0) return HSK_OK;
    const int G = user_group ? n_groups : 0;
    det_metric_sums_kernel<<<1 + G, 256, 0, as_stream(stream)>>>(per_user, Be, n_ks * 3, u_idx, user_group, G, sums);
    return check_launch("hsk_rank_metrics_sums_det");
}

extern "C" int hsk_rank_metrics_sums_det_pack(const float* per_user, int Be, int batch, int n_ks, const int64_t* u_idx,
                                              const int32_t* user_group, int n_groups, int n_trials, const int32_t* active,
                                              int n_active, double* sums, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(per_user && u_idx && sums, "hsk_rank_metrics_sums_det_pack: null pointer");
    HSK_REQUIRE(n_ks >= 1 && n_ks <= 8 && n_groups >= 0 && Be >= 0 && batch >= 1,
                "hsk_rank_metrics_sums_det_pack: need 1 <= n_ks <= 8, batch >= 1");
    HSK_REQUIRE(n_trials >= 1 && n_active >= 0 && n_active <= n_trials && n_active <= 65535,
                "hsk_rank_metrics_sums_det_pack: need 0 <= n_active <= n_trials, n_trials >= 1, n_active <= 65535 (n_trials=%d n_active=%d)",
                n_trials, n_active);
    HSK_REQUIRE(n_active == 0 || active, "hsk_rank_metrics_sums_det_pack: active is null");
    if (Be == 0 || n_active == 0) return HSK_OK;
    const int G = user_group ? n_groups : 0;
    det_metric_sums_pack_kernel<<<dim3(1 + G, n_active), 256, 0, as_stream(stream)>>>(per_user, Be, batch, n_ks * 3, u_idx, user_group,
                                                                                    G, n_groups, active, n_trials, sums, status);
    return check_launch("hsk_rank_metrics_sums_det_pack");
}
