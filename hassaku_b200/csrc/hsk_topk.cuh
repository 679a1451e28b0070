// Top-k machinery shared by the evaluator kernels.
//
// A candidate is ONE 64-bit key:  (orderable(score) << 32) | (0xFFFFFFFF - item_id)
// so that a plain unsigned compare orders by score descending and, among equal scores, by item id ascending —
// a strict total order, which makes the result independent of tile / split / shard processing order (the
// reference's torch.topk leaves the order of ties implementation-defined, SURVEY §8c).  Key 0 = empty slot.
//
// Per row a list of up to kCap = 256 keys is kept; when it may overflow it is sorted by one warp with a
// register-resident bitonic network (8 keys per lane) and cut back to the best k.
#pragma once
#include "hsk_common.cuh"

namespace hsk {

constexpr int kCap = 256;          // candidate-list capacity per row
constexpr int kKeysPerLane = 8;    // kCap / 32
constexpr int kMaxK = 128;         // largest supported k (K_VALUES max is 100, eval/eval.py:20)

// -0 is mapped to +0 first: the two compare equal, so they are one score and tie by item id
__device__ __forceinline__ uint32_t orderable(float f) {
    uint32_t u = __float_as_uint(f);
    u = (u == 0x80000000u) ? 0u : u;
    return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float from_orderable(uint32_t o) {
    uint32_t u = o ^ ((o >> 31) ? 0x80000000u : 0xFFFFFFFFu);
    return __uint_as_float(u);
}
__device__ __forceinline__ uint64_t make_key(float score, uint32_t id) {
    return (static_cast<uint64_t>(orderable(score)) << 32) | static_cast<uint64_t>(0xFFFFFFFFu - id);
}
__device__ __forceinline__ float key_score(uint64_t key) { return from_orderable(static_cast<uint32_t>(key >> 32)); }
__device__ __forceinline__ int32_t key_id(uint64_t key) {
    return key == 0 ? -1 : static_cast<int32_t>(0xFFFFFFFFu - static_cast<uint32_t>(key & 0xFFFFFFFFu));
}

// Sort 32 * KPL keys held by a warp (element e = r * 32 + lane lives in key[r] of `lane`) in DESCENDING order.
template <int KPL>
__device__ __forceinline__ void warp_sort_desc(uint64_t (&key)[KPL], int lane) {
    // log2-indexed unit-stride loops: nvcc fully unrolls them, so key[] stays in registers (with shift-stepped loops it
    // did not, and the network ran out of local memory: ~130 k cycles per 512-key sort, measured)
    constexpr int LOGN = (KPL == 1 ? 5 : KPL == 2 ? 6 : KPL == 4 ? 7 : KPL == 8 ? 8 : 9);
    static_assert((32 * KPL) == (1 << LOGN), "KPL must be a power of two <= 16");
#pragma unroll
    for (int lk = 1; lk <= LOGN; ++lk) {
#pragma unroll
        for (int lj = LOGN - 1; lj >= 0; --lj) {
            if (lj < lk) {
                const int k = 1 << lk, j = 1 << lj;
                if (lj >= 5) {
                    const int jr = j >> 5;
#pragma unroll
                    for (int r = 0; r < KPL; ++r) {
                        if ((r & jr) == 0) {
                            const int rp = r | jr;
                            const bool desc = (((r * 32 + lane) & k) == 0);
                            const uint64_t a = key[r], b = key[rp];
                            const bool sw = desc ? (a < b) : (a > b);
                            key[r] = sw ? b : a;
                            key[rp] = sw ? a : b;
                        }
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < KPL; ++r) {
                        const uint64_t other = __shfl_xor_sync(kFull, key[r], j);
                        const bool lower = (lane & j) == 0;
                        const bool desc = (((r * 32 + lane) & k) == 0);
                        const bool keep_max = (lower == desc);
                        const uint64_t mx = key[r] > other ? key[r] : other;
                        const uint64_t mn = key[r] > other ? other : key[r];
                        key[r] = keep_max ? mx : mn;
                    }
                }
            }
        }
    }
}

// element #pos (0 <= pos < 256) of a warp-held sorted list, broadcast to every lane
template <int KPL>
__device__ __forceinline__ uint64_t warp_list_at(const uint64_t (&key)[KPL], int pos) {
    uint64_t v = 0;
#pragma unroll
    for (int r = 0; r < KPL; ++r)
        if (r == (pos >> 5)) v = key[r];
    return __shfl_sync(kFull, v, pos & 31);
}

// membership test in a sorted int32 range [lo, hi) (one CSR row): lower_bound + compare
__device__ __forceinline__ bool csr_contains(const int32_t* __restrict__ idx, int64_t lo, int64_t hi, int32_t x) {
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(idx + mid) < x) lo = mid + 1; else hi = mid;
    }
    return lo < end && __ldg(idx + lo) == x;
}

// KPL membership tests in lock-step: every step of the binary search issues KPL independent loads per lane, so the
// latencies of the searches overlap (one after the other they cost KPL x log2(len) dependent global-memory round trips —
// measured 125 k cycles per list cut in the tensor-core evaluator).  found[r] = id[r] is in the sorted row [lo, hi).
template <int KPL>
__device__ __forceinline__ void csr_contains_many(const int32_t* __restrict__ idx, int64_t lo, int64_t hi, const int32_t (&id)[KPL],
                                                  const bool (&active)[KPL], bool (&found)[KPL]) {
    const int len = (int)(hi - lo);
    const int32_t* row = idx + lo;
    int pos[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) pos[r] = 0;
    int step = 1;
    while (step * 2 <= len) step *= 2;
    for (; step > 0; step >>= 1) {
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            const int probe = pos[r] + step;
            if (active[r] && probe <= len && __ldg(row + probe - 1) < id[r]) pos[r] = probe;
        }
    }
#pragma unroll
    for (int r = 0; r < KPL; ++r) found[r] = active[r] && pos[r] < len && __ldg(row + pos[r]) == id[r];
}

// Membership of KPL ids per lane in a SHORT sorted row the other way round: the row is read once, coalesced (32 ids per
// round), and every id of it is broadcast to the warp and compared with the lane's KPL register-resident candidates —
// len * KPL compares per lane but a single global-memory round trip per 32 row entries, instead of log2(len) dependent
// round trips per candidate.  Use for rows up to a few hundred entries.
template <int KPL>
__device__ __forceinline__ void csr_contains_bcast(const int32_t* __restrict__ idx, int64_t lo, int64_t hi, const int32_t (&id)[KPL],
                                                   bool (&found)[KPL], int lane) {
#pragma unroll
    for (int r = 0; r < KPL; ++r) found[r] = false;
    for (int64_t base = lo; base < hi; base += 32) {
        const int32_t x = (base + lane < hi) ? __ldg(idx + base + lane) : -2;
        const int cntr = (int)min((int64_t)32, hi - base);
        for (int j = 0; j < cntr; ++j) {
            const int32_t xj = __shfl_sync(kFull, x, j);
#pragma unroll
            for (int r = 0; r < KPL; ++r) found[r] |= (id[r] == xj);
        }
    }
}

// Cut a row's candidate list (n <= kCap keys at `list`, global or shared memory) back to its best k, sorted.
// Returns the new length min(n, k); *thr_key receives the k-th key (0 while the list holds fewer than k).
template <int KPL = kKeysPerLane>
__device__ __forceinline__ int warp_prune_list(uint64_t* list, int n, int k, int lane, uint64_t* thr_key) {
    uint64_t key[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int e = r * 32 + lane;
        key[r] = (e < n) ? list[e] : 0ull;
    }
    warp_sort_desc<KPL>(key, lane);
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int e = r * 32 + lane;
        if (e < k) list[e] = key[r];
    }
    *thr_key = (n >= k) ? warp_list_at<KPL>(key, k - 1) : 0ull;
    return n < k ? n : k;
}

// Same, applying the exclusion mask lazily: entries [n_checked, n) have not been tested against the user's exclusion row
// yet (the scoring epilogues append raw candidates so that their hot loop has no dependent global loads); an excluded
// item is re-keyed to score -inf (eval/eval.py:250-251) before the sort.  The 8 binary searches of a lane are
// independent, so their latencies overlap.
template <int KPL = kKeysPerLane>
__device__ __forceinline__ int warp_prune_list_masked(uint64_t* list, int n, int n_checked, int k, int lane, uint64_t* thr_key,
                                                      const int32_t* __restrict__ excl, int64_t lo, int64_t hi,
                                                      unsigned long long* tprof = nullptr) {
    long long t0 = tprof ? clock64() : 0;
    uint64_t key[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int e = r * 32 + lane;
        key[r] = (e < n) ? list[e] : 0ull;
    }
    if (tprof) { uint64_t x = 0; for (int r = 0; r < KPL; ++r) x ^= key[r]; if (x == 0x1234567ull) list[0] = x; const long long t1 = clock64(); tprof[0] += t1 - t0; t0 = t1; }
    if (hi > lo) {
        int32_t id[KPL];
        bool active[KPL], found[KPL];
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            const int e = r * 32 + lane;
            active[r] = e >= n_checked && e < n;
            id[r] = key_id(key[r]);
        }
        csr_contains_many<KPL>(excl, lo, hi, id, active, found);
#pragma unroll
        for (int r = 0; r < KPL; ++r)
            if (found[r]) key[r] = make_key(-INFINITY, (uint32_t)id[r]);
    }
    if (tprof) { uint64_t x = 0; for (int r = 0; r < KPL; ++r) x ^= key[r]; if (x == 0x1234567ull) list[0] = x; const long long t1 = clock64(); tprof[1] += t1 - t0; t0 = t1; }
    warp_sort_desc<KPL>(key, lane);
    if (tprof) { uint64_t x = 0; for (int r = 0; r < KPL; ++r) x ^= key[r]; if (x == 0x1234567ull) list[0] = x; const long long t1 = clock64(); tprof[2] += t1 - t0; t0 = t1; }
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int e = r * 32 + lane;
        if (e < k) list[e] = key[r];
    }
    if (tprof) { const long long t1 = clock64(); tprof[3] += t1 - t0; tprof[4] += 1; }
    *thr_key = (n >= k) ? warp_list_at<KPL>(key, k - 1) : 0ull;
    return n < k ? n : k;
}

// Cut a CONTIGUOUS candidate list (n <= 32 * KPL keys) back to ~k without sorting: exclusion test of the entries beyond
// n_checked (lock-step binary searches), radix select on the 16 most significant key bits for the largest prefix T with
// count(prefix >= T) >= k, compaction of the survivors (k plus the ties of bucket T) to list[0..total).  The new
// threshold is the lower edge of bucket T — conservative, the exact order is established once by the final sort.
// If the tie bucket is huge (degenerate scores) the cut falls back to the exact sort and keeps exactly k, with the
// exact k-th key as threshold.  Returns the number of survivors (<= max_keep).
template <int KPL>
__device__ __forceinline__ int warp_cut_list(uint64_t* list, int n, int n_checked, int k, int max_keep, int lane,
                                             const int32_t* __restrict__ excl, int64_t lo, int64_t hi, float* new_tau,
                                             uint64_t* new_taukey) {
    uint64_t key[KPL];
    bool unchecked[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) {
        const int e = r * 32 + lane;
        key[r] = (e < n) ? list[e] : 0ull;
        unchecked[r] = e >= n_checked && e < n;
    }
    if (hi > lo) {
        int32_t id[KPL];
        bool found[KPL];
#pragma unroll
        for (int r = 0; r < KPL; ++r) id[r] = key_id(key[r]);
        csr_contains_many<KPL>(excl, lo, hi, id, unchecked, found);
#pragma unroll
        for (int r = 0; r < KPL; ++r)
            if (found[r]) key[r] = make_key(-INFINITY, (uint32_t)id[r]);
    }
    uint32_t T = 0;
    if (n > k) {
        uint32_t pre[KPL];
#pragma unroll
        for (int r = 0; r < KPL; ++r) pre[r] = (uint32_t)(key[r] >> 48);
#pragma unroll 1
        for (int b = 15; b >= 0; --b) {
            const uint32_t cand = T | (1u << b);
            int c = 0;
#pragma unroll
            for (int r = 0; r < KPL; ++r) c += (pre[r] >= cand) ? 1 : 0;
            c = __reduce_add_sync(kFull, c);
            if (c >= k) T = cand;
        }
    }
    int mine = 0;
#pragma unroll
    for (int r = 0; r < KPL; ++r) mine += (key[r] != 0ull && (uint32_t)(key[r] >> 48) >= T) ? 1 : 0;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += up;
    }
    const int total = __shfl_sync(kFull, incl, 31);
    if (total > max_keep) {
        warp_sort_desc<KPL>(key, lane);
#pragma unroll
        for (int r = 0; r < KPL; ++r) {
            const int e = r * 32 + lane;
            if (e < k) list[e] = key[r];
        }
        const uint64_t thr = warp_list_at<KPL>(key, k - 1);
        *new_taukey = thr;
        *new_tau = key_score(thr);
        return k;
    }
    int pos = incl - mine;
#pragma unroll
    for (int r = 0; r < KPL; ++r)
        if (key[r] != 0ull && (uint32_t)(key[r] >> 48) >= T) list[pos++] = key[r];
    *new_tau = (n > k) ? from_orderable(T << 16) : -INFINITY;
    *new_taukey = (n > k) ? ((uint64_t)(T << 16) << 32) : 0ull;
    return total;
}

// hsk_eval.cu: merge of n_lists sorted key lists per row laid out [list][row][stride] (split plans of the eval kernels)
int launch_merge_keys(const uint64_t* lists, int n_lists, int rows, int stride, int k, float* out_scores, int32_t* out_ids, cudaStream_t s,
                      const float* Ub, const float* Gb, const int64_t* u_idx, int64_t n_users);

}  // namespace hsk
