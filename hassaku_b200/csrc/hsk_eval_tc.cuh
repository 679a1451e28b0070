// Pieces shared by the tensor-core evaluator kernels (hsk_eval_tc.cu: one CTA per 128-user tile, cta_group::1;
// hsk_eval_tc2.cu: CTA pairs, cta_group::2): tile constants, the argument block, tcgen05 / TMA / mbarrier wrappers, the
// candidate-list scan, cut and final sort.
#pragma once
#include <cuda.h>
#include <stdlib.h>
#include <cuda_bf16.h>

#include "hsk_topk.cuh"

namespace hsk {

constexpr int TC_BM = 128;        // users per CTA tile (UMMA_M)
constexpr int TC_BN = 128;        // items per tile (UMMA_N)
constexpr int TC_KB_BYTES = 128;  // bytes of K per k-block (one 128B swizzle atom)
constexpr int TC_MAX_STAGES = 10;          // B-tile ring depth is chosen at launch: as many 16 KB stages as fit beside the A tile
constexpr int TC_TILE_BYTES = TC_BN * TC_KB_BYTES;  // 16 KB per operand tile per k-block
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_THREADS = 64 + TC_EPI_WARPS * 32;   // TMA warp + MMA warp + 8 epilogue warps
constexpr int TC_ACC_STAGES = 4;           // accumulator stages in TMEM: 4 x 128 fp32 columns = all 512 columns
constexpr int TC_KPL = 16;                 // candidate keys per lane in the epilogue lists
constexpr int TC_CAP = 32 * TC_KPL;        // 512-entry lists: a cut every ~(512 - 128 - k) appends instead of ~28
constexpr int kMaxItemShards = 8;  // = HSK_MAX_PEERS
constexpr int TC_MAX_KB = 8;      // kpad * elem_size <= 1024 bytes -> d <= 512 (bf16) / 256 (tf32)

struct EvalTcArgs {
    const float* __restrict__ Ub;   // user bias TABLE (indexed by u_idx) or null
    const float* __restrict__ Ib;   // local item bias or null
    const float* __restrict__ Gb;
    const int64_t* __restrict__ u_idx;
    const int64_t* __restrict__ u_rows;   // row of the Ub table per batch entry (null: = u_idx)
    const int64_t* __restrict__ excl_indptr;
    const int32_t* __restrict__ excl_indices;
    int64_t n_users, n_local, id_offset, id_stride;
    int Be, k, num_kb, kelems_per_kb;
    int n_tiles, tiles_per_split, n_splits, n_stages;
    uint64_t* cand;
    float* out_scores;
    int32_t* out_ids;
    int32_t* status;
    // item SHARDS behind one launch of the CTA-pair kernel (hsk_eval_topk_tc_shards; 1 = one table): shard q holds the items
    // q + n_shards * row, its rows are tiles [shard_tile_end[q - 1], shard_tile_end[q]) of the launch, walked shard by shard
    int n_shards;
    int shard_tile_end[kMaxItemShards];
    int64_t shard_rows[kMaxItemShards];
    const float* shard_Ib[kMaxItemShards];
};
struct EvalTcMaps {                 // the shards' packed tables (one TMA descriptor each)
    CUtensorMap m[kMaxItemShards];
};

// ---- PTX wrappers ----
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
                     "r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
template <bool TF32>
__device__ __forceinline__ void tc_mma(uint32_t tmem_c, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (TF32) {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::
                         "r"(tmem_c), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                     : "memory");
    } else {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::
                         "r"(tmem_c), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                     : "memory");
    }
}
__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, version 1 = sm_100):
// start address >> 4 | SBO = 1024 B (8 rows x 128 B) | layout type 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void tc_st32(uint32_t taddr, const float (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(taddr),
        "f"(r[0]), "f"(r[1]), "f"(r[2]), "f"(r[3]), "f"(r[4]), "f"(r[5]), "f"(r[6]), "f"(r[7]), "f"(r[8]), "f"(r[9]), "f"(r[10]),
        "f"(r[11]), "f"(r[12]), "f"(r[13]), "f"(r[14]), "f"(r[15]), "f"(r[16]), "f"(r[17]), "f"(r[18]), "f"(r[19]), "f"(r[20]),
        "f"(r[21]), "f"(r[22]), "f"(r[23]), "f"(r[24]), "f"(r[25]), "f"(r[26]), "f"(r[27]), "f"(r[28]), "f"(r[29]), "f"(r[30]),
        "f"(r[31])
        : "memory");
}
__device__ __forceinline__ void tc_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ float fmax3(float a, float b, float c) {   // FMNMX3 (sm_100)
    float d;
    asm("max.f32 %0, %1, %2, %3;\n" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// The item-bias row of NCHUNK x 32 consecutive items -> TMEM columns [taddr, +NCHUNK * 32) of this thread's lane (every lane =
// user row gets the same values).  The MMA of that tile then accumulates on top (enable_input_d = 1), so the epilogue reads
// score' = bias + <u, v> straight from the accumulator: no bias add in the hot loop.  `sb` = the bias values in SHARED memory
// (staged one tile ahead by the pair, so no global-memory latency sits between reading a stage and releasing it); the
// loads are warp-uniform 128-bit broadcasts.
template <int NCHUNK>
__device__ __forceinline__ void tc_write_bias(const float* sb, uint32_t taddr) {
#pragma unroll 1
    for (int c = 0; c < NCHUNK; ++c) {
        float b[32];
        const float4* p4 = reinterpret_cast<const float4*>(sb + c * 32);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const float4 x = p4[q];
            b[4 * q + 0] = x.x; b[4 * q + 1] = x.y; b[4 * q + 2] = x.z; b[4 * q + 3] = x.w;
        }
        tc_st32(taddr + (uint32_t)(c * 32), b);
    }
    tc_st_wait();
}

// ---- the user's exclusion row as a CURSOR: a thread meets its candidates in ascending item-id order (tiles, chunks and
// elements are all walked upwards), and the CSR row is sorted, so "is this id excluded?" is a comparison with the next
// unconsumed exclusion — the mask of eval/eval.py:250-251 is applied at the append, exactly, with <= n_excl dependent loads
// per thread over the whole sweep.  (Round 1 kept raw candidates and tested them at the list cuts with lock-step binary
// searches, which forced the lists to hold k + n_excl entries and made every cut ~5x more expensive.)
struct ExCursor {
    const int32_t* __restrict__ idx;
    int64_t pos, hi;
    uint32_t next;          // indices[pos], or 0xFFFFFFFF when the row is used up
};
__device__ __forceinline__ void ex_init(ExCursor& c, const int32_t* __restrict__ idx, int64_t lo, int64_t hi) {
    c.idx = idx; c.pos = lo; c.hi = hi;
    c.next = lo < hi ? (uint32_t)__ldg(idx + lo) : 0xFFFFFFFFu;
}
__device__ __forceinline__ bool ex_excluded(ExCursor& c, uint32_t gid) {
    while (c.next < gid) {
        ++c.pos;
        c.next = c.pos < c.hi ? (uint32_t)__ldg(c.idx + c.pos) : 0xFFFFFFFFu;
    }
    return c.next == gid;
}

// Epilogue of one 32-column chunk for one row: v[] holds score' = item bias + dot (the per-row user / global bias does not
// change the ranking inside a row and is added when the final scores are written).  `region` is this thread's PRIVATE
// half of the row's candidate list, so an append is a register increment and a fire-and-forget store.
// tc_chunk_max: 8 group maxima of 4 (FMNMX3 + FMNMX each) and their maximum (NaN = a column beyond the table: ignored by
// max).  tc_scan_groups: only the groups whose maximum reaches the row's threshold are looked at — per row-chunk a
// survivor is rare (~6 %), but per WARP (32 rows with their own thresholds) some lane almost always has one, so this
// divergent path is the common path and its length, not the all-clear path, sets the epilogue's cost.
__device__ __forceinline__ float tc_chunk_max(const float (&v)[32], float (&g)[8]) {
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] = fmaxf(fmax3(v[4 * j], v[4 * j + 1], v[4 * j + 2]), v[4 * j + 3]);
    return fmax3(fmax3(g[0], g[1], g[2]), fmax3(g[3], g[4], g[5]), fmaxf(g[6], g[7]));
}
// Kept compact and branch-poor on purpose.  Measured alternatives (18 944 users x 1 M items x 256, bf16, one-CTA kernel):
//   one guarded append block per element, fully unrolled (105 KB of kernel body)                 34.3 ms
//   warp-uniform vote per group (8 x __any_sync + branch per chunk, group values as named registers)  14.6 ms
//   this version: an 8-bit mask of the groups whose maximum reaches the threshold (8 compares), then per set bit the group's
//   4 values pulled out of the register array by a 3-level select tree (28 selects, no local memory)   10.7 ms
// — every taken branch in this divergent path costs an instruction-fetch bubble, selects do not.
// `nvalid`: columns of the chunk that exist (32 except in the table's ragged last tile, whose missing rows TMA fills with
// zeros: their scores are never candidates).  The bound is applied HERE, at the append, so that the hot path reads the
// accumulator registers in place (patching the chunk's values instead cost 32 register moves per chunk).
__device__ __forceinline__ void tc_scan_groups(const float (&v)[32], const float (&g)[8], float tau, uint64_t taukey, uint32_t gid0,
                                               uint32_t id_stride, int& cnt, uint64_t* region, ExCursor& ex, int nvalid) {
    uint32_t gm = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) gm |= (g[j] >= tau) ? (1u << j) : 0u;
    while (gm) {
        const int j = __ffs(gm) - 1;
        gm &= gm - 1;
        float a16[16], a8[8], a4[4];
#pragma unroll
        for (int i = 0; i < 16; ++i) a16[i] = (j & 4) ? v[16 + i] : v[i];
#pragma unroll
        for (int i = 0; i < 8; ++i) a8[i] = (j & 2) ? a16[8 + i] : a16[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) a4[i] = (j & 1) ? a8[4 + i] : a8[i];
        uint32_t em = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) em |= (a4[q] >= tau) ? (1u << q) : 0u;
        while (em) {
            const int q = __ffs(em) - 1;
            em &= em - 1;
            const float x = (q & 2) ? ((q & 1) ? a4[3] : a4[2]) : ((q & 1) ? a4[1] : a4[0]);
            const uint32_t gid = gid0 + (uint32_t)(4 * j + q) * id_stride;
            const uint64_t key = make_key(x, gid);
            if (key > taukey && 4 * j + q < nvalid && !ex_excluded(ex, gid)) region[cnt++] = key;
        }
    }
}

constexpr int TC_HALF_CAP = TC_CAP / 2;   // 256 entries per column half (two-region layout)

// A row's candidate list of TC_CAP = 512 keys is split into NR regions (one per epilogue warp that shares the row: NR = 2
// column halves, or 4 column quarters), region q at lp[q * (TC_CAP / NR) ..) with c[q] entries.
//
// tc_cut_row: cut the list back to ~k WITHOUT sorting: a radix select on the 16 most significant bits of the keys finds
// the largest prefix T with count(prefix >= T) >= k; everything below T is dropped, the survivors (k plus the few ties of the
// T bucket) are compacted and dealt round-robin to the regions (survivor #pos -> region pos % NR, slot pos / NR).  The new
// threshold is the lower edge of bucket T — conservative, so no top-k item is ever lost; the exact order is established
// once, by the final sort.  ~1.5 k cycles instead of ~56 k for the 512-key bitonic network.  Every entry is an admissible
// item (exclusions are dropped at the append).  Returns the number of survivors; region q then holds
// (total - q + NR - 1) / NR of them.
template <int NR>
static __device__ __noinline__ int tc_cut_row(uint64_t* lp, const int* c, int k, int lane, int max_keep, float* new_tau,
                                              uint64_t* new_taukey) {
    constexpr int RC = TC_CAP / NR;
    uint64_t key[TC_KPL];
    int n = 0;
#pragma unroll
    for (int q = 0; q < NR; ++q) n += c[q];
#pragma unroll
    for (int r = 0; r < TC_KPL; ++r) {
        const int e = r * 32 + lane;
        const int q = e / RC, idx = e % RC;
        key[r] = (idx < c[q]) ? lp[e] : 0ull;
    }
    uint32_t T = 0;
    if (n > k) {
        uint32_t pre[TC_KPL];
#pragma unroll
        for (int r = 0; r < TC_KPL; ++r) pre[r] = (uint32_t)(key[r] >> 48);   // empty slots have prefix 0
#pragma unroll 1
        for (int b = 15; b >= 0; --b) {
            const uint32_t cand = T | (1u << b);
            int cc = 0;
#pragma unroll
            for (int r = 0; r < TC_KPL; ++r) cc += (pre[r] >= cand) ? 1 : 0;
            cc = __reduce_add_sync(kFull, cc);
            if (cc >= k) T = cand;
        }
    }
    // compaction: keep keys whose prefix >= T (all valid keys when n <= k)
    int mine = 0;
#pragma unroll
    for (int r = 0; r < TC_KPL; ++r) mine += (key[r] != 0ull && (uint32_t)(key[r] >> 48) >= T) ? 1 : 0;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += up;
    }
    const int total = __shfl_sync(kFull, incl, 31);
    if (total > max_keep) {
        // degenerate score distribution (a huge tie bucket, e.g. all-equal scores): exact cut by the full sort; ties are
        // then resolved by the strict key order (lower item id wins), which the scan honours through `taukey`
        warp_sort_desc<TC_KPL>(key, lane);
#pragma unroll
        for (int r = 0; r < TC_KPL; ++r) {
            const int e = r * 32 + lane;
            if (e < k) lp[(e % NR) * RC + e / NR] = key[r];
        }
        const uint64_t thr = warp_list_at<TC_KPL>(key, k - 1);
        *new_taukey = thr;
        *new_tau = key_score(thr);
        return k;
    }
    int pos = incl - mine;
#pragma unroll
    for (int r = 0; r < TC_KPL; ++r) {
        if (key[r] != 0ull && (uint32_t)(key[r] >> 48) >= T) {
            lp[(pos % NR) * RC + pos / NR] = key[r];
            ++pos;
        }
    }
    *new_tau = (n > k) ? from_orderable(T << 16) : -INFINITY;   // lower edge of bucket T (n > k implies T >= 0x007F)
    *new_taukey = (n > k) ? ((uint64_t)(T << 16) << 32) : 0ull;
    return total;
}

// The -inf tail of a row with fewer than k admissible items (total < k survivors after the last cut): the reference ranks
// the user's excluded items after every admissible one, at score -inf, lowest id first.  The scan never appends them, so
// the warp walks the exclusion row [lo, hi) upwards from the first id >= id_lo and appends, after the survivors in the
// round-robin layout, the first k ids that this launch covers (`covered(id)`; the walk stops past id_hi), keyed
// make_key(-inf, id).  k of them rather than k - total keeps the result exact when admissible items score -inf too.
// Returns the new list length (<= total + k < 256 for the final sort).
template <int NR, class Covered>
static __device__ __forceinline__ int tc_fill_excluded(uint64_t* lp, int total, int k, int lane, const int32_t* __restrict__ excl,
                                                       int64_t lo, int64_t hi, uint32_t id_lo, uint32_t id_hi, Covered covered) {
    constexpr int RC = TC_CAP / NR;
    {   // lower bound of id_lo in the sorted row
        int64_t a = lo, b = hi;
        while (a < b) {
            const int64_t mid = (a + b) >> 1;
            if ((uint32_t)__ldg(excl + mid) < id_lo) a = mid + 1; else b = mid;
        }
        lo = a;
    }
    int added = 0;
    for (int64_t base = lo; base < hi && added < k; base += 32) {
        const int64_t p = base + lane;
        const uint32_t id = p < hi ? (uint32_t)__ldg(excl + p) : 0xFFFFFFFFu;
        const bool take = p < hi && id <= id_hi && covered(id);
        const unsigned m = __ballot_sync(kFull, take);
        const int pos = added + __popc(m & ((1u << lane) - 1));
        if (take && pos < k) {
            const int e = total + pos;
            lp[(e % NR) * RC + e / NR] = make_key(-INFINITY, id);
        }
        added += __popc(m);
        if (__any_sync(kFull, id > id_hi)) break;
    }
    __syncwarp();
    return total + min(added, k);
}

// Final, exact: `total` <= 255 keys dealt round-robin over the NR regions (as tc_cut_row and tc_fill_excluded leave them)
// are sorted with the 256-key network and the best k written to lp[0..k) / returned in key[] (element e = r * 32 + lane).
template <int NR>
static __device__ __noinline__ void tc_final_sort(uint64_t* lp, int total, int k, int lane, uint64_t (&key)[kKeysPerLane]) {
    constexpr int RC = TC_CAP / NR;
#pragma unroll
    for (int r = 0; r < kKeysPerLane; ++r) {
        const int e = r * 32 + lane;
        key[r] = (e < total) ? lp[(e % NR) * RC + e / NR] : 0ull;
    }
    warp_sort_desc<kKeysPerLane>(key, lane);
    __syncwarp();
#pragma unroll
    for (int r = 0; r < kKeysPerLane; ++r) {
        const int e = r * 32 + lane;
        if (e < k) lp[e] = key[r];
    }
}

}  // namespace hsk
