// Full-rank evaluator, tensor-core mode (TF32 / BF16): scores = U_b · V^T on tcgen05 with TMEM accumulators, fed by TMA,
// fused with bias add, exclusion mask and running top-k — the [Be, I] score matrix never leaves the SM.
//
// Per CTA (320 threads, 1 per SM):
//   warp 0      TMA producer: the 128-user A tile is loaded ONCE (resident for every item tile); item (B) tiles of
//               128 rows x 128 bytes of K stream through a ring of up to 10 stages (cp.async.bulk.tensor.2d, SWIZZLE_128B)
//   warp 1      allocates all 512 TMEM columns (4 accumulator stages x 128 fp32 columns) and issues tcgen05.mma
//               (cta_group::1, M = 128, N = 128, 32 bytes of K per instruction), tcgen05.commit -> mbarriers
//   warps 2-9   epilogue (two warps per scheduler): a thread owns accumulator lane (= user row) r and one 64-column half of
//               the tile; tcgen05.ld 32 columns at a time, + item bias (128-bit uniform loads), chunk max against the row's
//               running k-th score; only survivors are keyed and appended to the row's candidate list (shared-memory
//               counter); the exclusion mask is applied lazily when a list is cut back by the warp-cooperative bitonic
//               sort (hsk_topk.cuh).  The accumulator stage is released before the pruning so the MMA of tile t+1
//               overlaps the epilogue of tile t.
// Operands are packed row-major [rows, kpad] (K-major for both A and B) by hsk_pack_rows: bf16 (round-to-nearest-even)
// or tf32 (fp32 container, rna-rounded), zero padded to a multiple of 128 bytes of K.
#include "hsk_eval_tc.cuh"

namespace hsk {

template <bool TF32>
__global__ void __launch_bounds__(TC_THREADS, 1)
eval_topk_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, EvalTcArgs a) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ uint64_t bar_full[TC_MAX_STAGES], bar_empty[TC_MAX_STAGES], bar_a, bar_tfull[TC_ACC_STAGES], bar_tempty[TC_ACC_STAGES];
    __shared__ uint32_t s_tmem_base;
    // per-row top-k state shared by the two epilogue warps of a row (column halves)
    __shared__ float s_tau[TC_BM];
    __shared__ uint64_t s_taukey[TC_BM];
    __shared__ int s_cnt2[2][TC_BM];   // per column half: entries of the row's candidate list
    __shared__ int64_t s_exlo[TC_BM], s_exhi[TC_BM];
    __shared__ float s_base[TC_BM];
    __shared__ int s_rowok[TC_BM];
    __shared__ int s_need[4][2][2];   // per pair / column half / tile parity: a list of this warp may overflow
    // per pair: item-bias tiles of the next tiles (ring of 2 x TC_ACC_STAGES... see the epilogue), written one tile ahead
    __shared__ __align__(16) float s_ib[4][2][TC_BN];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.x * TC_BM;
    const int split = blockIdx.y;
    const int t_begin = split * a.tiles_per_split;
    const int t_end = min(a.n_tiles, t_begin + a.tiles_per_split);
    const int n_my_tiles = t_end - t_begin;

    // 1024-byte aligned carve-up (SWIZZLE_128B atoms are 1024 B)
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* smA = smem;                                        // num_kb x 16 KB, resident
    unsigned char* smB = smem + (size_t)a.num_kb * TC_TILE_BYTES;     // n_stages x 16 KB

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.n_stages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
        mbar_init(&bar_a, 1);
        for (int s = 0; s < TC_ACC_STAGES; ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], TC_EPI_WARPS); }
        mbar_fence_init();
    }
    if (warp == 1) {  // TMEM: 2 accumulator stages x 128 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&s_tmem_base)), "n"(TC_ACC_STAGES * TC_BN));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::);
    }
    if (threadIdx.x >= 64 && threadIdx.x < 64 + TC_BM) {  // per-row state
        const int r = threadIdx.x - 64;
        const int row = m0 + r;
        int ok = 0;
        int64_t lo = 0, hi = 0;
        float base = 0.f;
        if (row < a.Be) {
            const int64_t u = a.u_idx[row];
            if (bad_index(u, a.n_users)) {
                if (a.status) atomicOr(a.status, HSK_STATUS_BAD_INDEX);
            } else {
                ok = 1;
                if (a.excl_indptr) { lo = a.excl_indptr[u]; hi = a.excl_indptr[u + 1]; }
                if (a.Ub) base += a.Ub[a.u_rows ? a.u_rows[row] : u];
            }
        }
        if (a.Gb) base += a.Gb[0];
        s_rowok[r] = ok; s_exlo[r] = lo; s_exhi[r] = hi; s_base[r] = base;
        s_tau[r] = -INFINITY; s_taukey[r] = 0ull;
        s_cnt2[0][r] = s_cnt2[1][r] = 0;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = s_tmem_base;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA));
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB));
            mbar_expect_tx(&bar_a, (uint32_t)a.num_kb * TC_TILE_BYTES);
            for (int kb = 0; kb < a.num_kb; ++kb) tma_load_2d(smA + (size_t)kb * TC_TILE_BYTES, &tmA, kb * a.kelems_per_kb, m0, &bar_a);
            int s = 0;
            uint32_t ph = 0;
            for (int t = 0; t < n_my_tiles; ++t) {
                const int n0 = (t_begin + t) * TC_BN;
                for (int kb = 0; kb < a.num_kb; ++kb) {
                    mbar_wait(&bar_empty[s], ph ^ 1u);
                    mbar_expect_tx(&bar_full[s], TC_TILE_BYTES);
                    tma_load_2d(smB + (size_t)s * TC_TILE_BYTES, &tmB, kb * a.kelems_per_kb, n0, &bar_full[s]);
                    if (++s == a.n_stages) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            // instruction descriptor: D = F32, A = B = BF16 (1) | TF32 (2), K-major both, N = 128, M = 128
            const uint32_t fmt = TF32 ? 2u : 1u;
            const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(TC_BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            mbar_wait(&bar_a, 0);
            tc_fence_after();
            int s = 0;
            uint32_t ph = 0;
            for (int t = 0; t < n_my_tiles; ++t) {
                const int as = t % TC_ACC_STAGES;
                mbar_wait(&bar_tempty[as], ((uint32_t)t / TC_ACC_STAGES) & 1u);   // the epilogue wrote this tile's bias row into the stage
                tc_fence_after();
                const uint32_t tmem_c = tmem_base + (uint32_t)as * TC_BN;
                for (int kb = 0; kb < a.num_kb; ++kb) {
                    mbar_wait(&bar_full[s], ph);
                    tc_fence_after();
                    const uint64_t da = umma_desc(smem_u32(smA + (size_t)kb * TC_TILE_BYTES));
                    const uint64_t db = umma_desc(smem_u32(smB + (size_t)s * TC_TILE_BYTES));
#pragma unroll
                    for (int k = 0; k < TC_KB_BYTES / 32; ++k)  // 32 bytes of K per MMA: advance the start address by 2 (x16 B)
                        tc_mma<TF32>(tmem_c, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, 1u);   // on top of the bias row
                    tc_commit(&bar_empty[s]);
                    if (++s == a.n_stages) { s = 0; ph ^= 1u; }
                }
                tc_commit(&bar_tfull[as]);
            }
        }
    } else {
        // ===== 8 epilogue warps: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4.  The two warps of a quarter
        // (a "pair", 64 threads) own the 32 rows of that quarter and synchronise only with each other. =====
        const int ew = warp - 2;
        const int quarter = warp & 3;
        const int half = ew >> 2;
        const int r = quarter * 32 + lane;   // row within the tile == TMEM lane
        const bool row_ok = s_rowok[r] != 0;
        uint64_t* list = a.cand + ((int64_t)split * a.Be + min(m0 + r, a.Be - 1)) * TC_CAP;
        const int prune_at = TC_HALF_CAP - TC_BN / 2;   // a tile appends at most 64 keys per column half
        uint64_t* region = list + half * TC_HALF_CAP;
        int cnt = 0;
        const int bar_id = 1 + quarter;
        const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 64);
        float* ib_pair = &s_ib[quarter][0][0];
        const int pt = half * 32 + lane;     // thread index within the pair (0..63)
        ExCursor ex;
        ex_init(ex, a.excl_indices, s_exlo[r], s_exhi[r]);
        // bias value of column `col` of tile `tt` (0 beyond the table / without item bias)
        auto ib_at = [&](int tt, int col) -> float {
            const int64_t n = (int64_t)(t_begin + tt) * TC_BN + col;
            return (a.Ib && tt < n_my_tiles && n < a.n_local) ? __ldg(a.Ib + n) : 0.f;
        };

        // prologue: the bias rows of the first TC_ACC_STAGES tiles go into the stages (through the pair's staging tile), the
        // stages to the MMA warp; then the staging slot of tile TC_ACC_STAGES is filled for the first loop iteration
        for (int ts = 0; ts < TC_ACC_STAGES && ts < n_my_tiles; ++ts) {
            ib_pair[pt] = ib_at(ts, pt);
            ib_pair[pt + 64] = ib_at(ts, pt + 64);
            named_bar_sync(bar_id, 64);
            tc_write_bias<2>(ib_pair + half * 64, tlane + (uint32_t)ts * TC_BN);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bar_tempty[ts]);
            named_bar_sync(bar_id, 64);
        }
        ib_pair[pt] = ib_at(TC_ACC_STAGES, pt);                 // slot 0 <- tile 4 (consumed at t = 0)
        ib_pair[pt + 64] = ib_at(TC_ACC_STAGES, pt + 64);
        named_bar_sync(bar_id, 64);

        int next_cut = 4;          // 128-item tiles after which every row is cut: 4, 6, 9, 13, ... (x 3 / 2)
        for (int t = 0; t < n_my_tiles; ++t) {
            const int as = t % TC_ACC_STAGES;
            const int64_t n0 = (int64_t)(t_begin + t) * TC_BN;
            const int ncols = (int)min((int64_t)TC_BN, a.n_local - n0);
            const float tau = s_tau[r];
            const uint64_t taukey = s_taukey[r];
            // the bias values the NEXT iteration writes (tile t + 5): in flight during this tile, stored before the pair barrier
            const float ibn0 = ib_at(t + 1 + TC_ACC_STAGES, pt), ibn1 = ib_at(t + 1 + TC_ACC_STAGES, pt + 64);
            mbar_wait(&bar_tfull[as], ((uint32_t)t / TC_ACC_STAGES) & 1u);
            tc_fence_after();
            const uint32_t taddr = tlane + (uint32_t)as * TC_BN;
            uint32_t raw0[32], raw1[32];
            tc_ld32_issue(taddr, raw0);
            tc_ld32_issue(taddr + 32u, raw1);
            tc_ld_wait();
            // both chunks are in registers: refill the stage with the bias row of tile t + 4 and release it right away
            if (t + TC_ACC_STAGES < n_my_tiles) {
                tc_write_bias<2>(ib_pair + (t & 1) * TC_BN + half * 64, taddr);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bar_tempty[as]);
            }
            {   // two inlined copies of the chunk body: chunk 0 reads raw0, chunk 1 reads raw1 in place
                auto chunk = [&](const uint32_t (&raw)[32], int cc) {
                    const int c = half * 64 + cc * 32;
                    if (c >= ncols) return;
                    float v[32], g[8];
#pragma unroll
                    for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(raw[e]);
                    const float mx = tc_chunk_max(v, g);
                    if (row_ok && mx >= tau)
                        tc_scan_groups(v, g, tau, taukey, (uint32_t)(a.id_offset + (n0 + c) * a.id_stride), (uint32_t)a.id_stride, cnt,
                                       region, ex, ncols - c);
                };
                chunk(raw0, 0);
                chunk(raw1, 1);
            }
            ib_pair[((t + 1) & 1) * TC_BN + pt] = ibn0;          // staging slot of tile t + 5, read after the pair barrier below
            ib_pair[((t + 1) & 1) * TC_BN + pt + 64] = ibn1;
            // Does any row of this pair need its list cut before the next tile?  Common case: no -> one flag store, one
            // pair barrier, one flag load per tile.  Only when a list may overflow (or at the last tile) do the two warps
            // exchange their counts and run the cut protocol (two more pair barriers).
            const bool last = (t + 1 == n_my_tiles);
            // scheduled cut of EVERY row after the same tiles (geometric schedule, see hsk_eval_tc2.cu); the fill trigger stays
            // as the safety net for score streams that are not in random order
            bool sched = false;
            if (t + 1 == next_cut) {
                sched = true;
                next_cut += next_cut / 2;
            }
            const bool warp_need = __any_sync(kFull, row_ok && cnt > prune_at) || last || sched;
            if (lane == 0) s_need[quarter][half][t & 1] = warp_need ? 1 : 0;
            named_bar_sync(bar_id, 64);
            const bool pair_need = (s_need[quarter][0][t & 1] | s_need[quarter][1][t & 1]) != 0;
            if (pair_need) {
                s_cnt2[half][r] = cnt;
                named_bar_sync(bar_id, 64);
                int my_a = 0, my_b = 0;
                bool my_need = false;
                if (lane < 16) {   // lane j looks at row j of this warp's 16 rows
                    const int rj = quarter * 32 + half * 16 + lane;
                    my_a = s_cnt2[0][rj];
                    my_b = s_cnt2[1][rj];
                    my_need = s_rowok[rj] && (my_a > prune_at || my_b > prune_at || last || sched);
                }
                unsigned need = __ballot_sync(kFull, my_need);
                while (need) {
                    const int j = __ffs(need) - 1;
                    need &= need - 1;
                    const int rr = quarter * 32 + half * 16 + j;
                    const int cA = __shfl_sync(kFull, my_a, j), cB = __shfl_sync(kFull, my_b, j);
                    uint64_t* lp = a.cand + ((int64_t)split * a.Be + (m0 + rr)) * TC_CAP;
                    float ntau;
                    uint64_t ntaukey;
                    // (a degenerate tie bucket makes tc_cut_row fall back to its exact sort and return exactly k survivors);
                    // intermediate cuts keep <= 160 of a half's 256 slots, the last one <= 192 in all for the final sort
                    const int cc[2] = {cA, cB};
                    const int total = tc_cut_row<2>(lp, cc, a.k, lane, last ? TC_HALF_CAP - TC_BN / 2 : 320, &ntau, &ntaukey);
                    __syncwarp();
                    const int nA = (total + 1) >> 1;
                    if (lane == 0) {
                        s_cnt2[0][rr] = nA; s_cnt2[1][rr] = total - nA;
                        s_tau[rr] = ntau; s_taukey[rr] = ntaukey;
                    }
                    if (last) {
                        int n_final = total;
                        if (total < a.k) {   // this split's items [t_begin, t_end) x TC_BN, local row n = global id id_offset + n * id_stride
                            const int64_t n_lo = (int64_t)t_begin * TC_BN, n_hi = min((int64_t)t_end * TC_BN, a.n_local) - 1;
                            n_final = tc_fill_excluded<2>(lp, total, a.k, lane, a.excl_indices, s_exlo[rr], s_exhi[rr],
                                                          (uint32_t)(a.id_offset + n_lo * a.id_stride),
                                                          (uint32_t)(a.id_offset + n_hi * a.id_stride),
                                                          [&](uint32_t id) { return ((int64_t)id - a.id_offset) % a.id_stride == 0; });
                        }
                        uint64_t keys[kKeysPerLane];
                        tc_final_sort<2>(lp, n_final, a.k, lane, keys);
                        if (a.n_splits == 1) {
                            const int64_t orow = (int64_t)(m0 + rr) * a.k;
                            const float base = s_base[rr];
#pragma unroll
                            for (int q = 0; q < kKeysPerLane; ++q) {
                                const int e = q * 32 + lane;
                                if (e < a.k) {
                                    a.out_scores[orow + e] = keys[q] ? key_score(keys[q]) + base : -INFINITY;
                                    a.out_ids[orow + e] = key_id(keys[q]);
                                }
                            }
                        }
                    }
                }
                named_bar_sync(bar_id, 64);
                cnt = s_cnt2[half][r];
            }
        }
        // rows with a bad user index: empty lists / -1 ids
        for (int j = 0; j < 16; ++j) {
            const int rr = quarter * 32 + half * 16 + j;
            if (m0 + rr < a.Be && !s_rowok[rr]) {
                if (a.n_splits == 1) {
                    for (int e = lane; e < a.k; e += 32) { a.out_scores[(int64_t)(m0 + rr) * a.k + e] = -INFINITY; a.out_ids[(int64_t)(m0 + rr) * a.k + e] = -1; }
                } else {
                    uint64_t* lp = a.cand + ((int64_t)split * a.Be + (m0 + rr)) * TC_CAP;
                    for (int e = lane; e < a.k; e += 32) lp[e] = 0ull;
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(TC_ACC_STAGES * TC_BN));
    }
}

// ---- operand packing: fp32 table rows (optionally gathered) -> [rows, kpad] bf16 | tf32, zero padded ----
template <bool TF32>
__global__ void __launch_bounds__(256) pack_rows_kernel(const float* __restrict__ src, int ld, int d, const int64_t* __restrict__ idx,
                                                        int64_t n_out, int64_t n_src, void* __restrict__ dst, int kpad, int32_t* status) {
    const int64_t total = n_out * kpad;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / kpad;
        const int k = (int)(e - r * kpad);
        float v = 0.f;
        if (k < d) {
            int64_t sr = idx ? idx[r] : r;
            if (bad_index(sr, n_src)) {
                if (status) atomicOr(status, HSK_STATUS_BAD_INDEX);
            } else {
                v = src[sr * ld + k];
            }
        }
        if (TF32) {
            uint32_t t;
            asm("cvt.rna.tf32.f32 %0, %1;\n" : "=r"(t) : "f"(v));
            reinterpret_cast<uint32_t*>(dst)[e] = t;
        } else {
            reinterpret_cast<__nv_bfloat16*>(dst)[e] = __float2bfloat16_rn(v);
        }
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_map(CUtensorMap* map, const void* base, bool tf32, int kpad, int64_t rows, int kelems_per_kb) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
        if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p)
            return set_err(HSK_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable: %s", cudaGetErrorString(e));
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    const size_t esz = tf32 ? 4 : 2;
    cuuint64_t dims[2] = {(cuuint64_t)kpad, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)kpad * esz};
    cuuint32_t box[2] = {(cuuint32_t)kelems_per_kb, (cuuint32_t)TC_BN};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, tf32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims,
                    strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_err(HSK_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return HSK_OK;
}

// `bn` = items per tile: TC_BN (one-CTA kernel) or 2 * TC_BN (CTA-pair kernel, whose row tiles come in pairs)
static void tc_plan_tiles(int Be, int nt, bool pair, int* n_tiles, int* tiles_per_split, int* n_splits) {
    int row_tiles = (Be + TC_BM - 1) / TC_BM;
    if (pair) row_tiles = (row_tiles + 1) / 2 * 2;
    const int want = sm_count();
    int splits = 1;
    if (row_tiles * 4 < want * 3) splits = (want + row_tiles - 1) / row_tiles;   // >= 75 % of the SMs busy: no split
    const int max_splits = nt / 8 > 0 ? nt / 8 : 1;   // at least 8 item tiles per split
    if (splits > max_splits) splits = max_splits;
    if (splits > 64) splits = 64;
    const int tps = (nt + splits - 1) / splits;
    *n_tiles = nt;
    *tiles_per_split = tps;
    *n_splits = (nt + tps - 1) / tps;
}
static void tc_plan(int Be, int64_t n_local, int bn, int* n_tiles, int* tiles_per_split, int* n_splits) {
    tc_plan_tiles(Be, (int)((n_local + bn - 1) / bn), bn > TC_BN, n_tiles, tiles_per_split, n_splits);
}

// hsk_eval_tc2.cu
int launch_eval_tc2(bool tf32, int row_tiles, int n_splits, size_t smem, cudaStream_t s, const CUtensorMap& tmA,
                    const EvalTcMaps& tmB, const EvalTcArgs& a);

}  // namespace hsk

using namespace hsk;

extern "C" int hsk_eval_tc_kpad(int d, int precision) {
    const int per_kb = (precision == HSK_PREC_TF32) ? 32 : 64;
    return ((d + per_kb - 1) / per_kb) * per_kb;
}

extern "C" int hsk_pack_rows(const float* src, int ld, int d, const int64_t* row_idx, int64_t n_out, int64_t n_src, void* dst,
                             int kpad, int precision, int32_t* status, hsk_stream_t stream) {
    HSK_REQUIRE(src && dst, "hsk_pack_rows: null pointer");
    HSK_REQUIRE(precision == HSK_PREC_TF32 || precision == HSK_PREC_BF16, "hsk_pack_rows: precision must be TF32 or BF16");
    HSK_REQUIRE(d >= 1 && ld >= d && kpad >= d && n_out >= 0, "hsk_pack_rows: bad sizes");
    if (n_out == 0) return HSK_OK;
    const int64_t total = n_out * kpad;
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (precision == HSK_PREC_TF32)
        pack_rows_kernel<true><<<(int)blocks, 256, 0, as_stream(stream)>>>(src, ld, d, row_idx, n_out, n_src, dst, kpad, status);
    else
        pack_rows_kernel<false><<<(int)blocks, 256, 0, as_stream(stream)>>>(src, ld, d, row_idx, n_out, n_src, dst, kpad, status);
    return check_launch("hsk_pack_rows");
}

extern "C" int64_t hsk_eval_topk_tc_scratch_bytes(int Be, int64_t n_local_items, int k) {
    (void)k;
    int nt, tps, ns1, ns2;     // enough for either kernel's split plan
    tc_plan(Be > 0 ? Be : 1, n_local_items > 0 ? n_local_items : 1, TC_BN, &nt, &tps, &ns1);
    tc_plan(Be > 0 ? Be : 1, n_local_items > 0 ? n_local_items : 1, 2 * TC_BN, &nt, &tps, &ns2);
    return (int64_t)(ns1 > ns2 ? ns1 : ns2) * (Be > 0 ? Be : 1) * TC_CAP * (int64_t)sizeof(uint64_t);
}

extern "C" int hsk_eval_topk_tc(const void* Uq, const void* Vq, int kpad, int precision, const float* Ub, const float* Ib,
                                const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be, int64_t n_users, int64_t n_local,
                                int64_t id_offset, int64_t id_stride, const int64_t* excl_indptr, const int32_t* excl_indices,
                                int k, float* top_scores, int32_t* top_ids, void* scratch, int64_t scratch_bytes,
                                int32_t* status, hsk_stream_t stream) {
    return hsk_eval_topk_tc_v(Uq, Vq, kpad, precision, Ub, Ib, Gb, u_idx, u_rows, Be, n_users, n_local, id_offset, id_stride,
                              excl_indptr, excl_indices, k, top_scores, top_ids, scratch, scratch_bytes, status, HSK_EVAL_TC_AUTO,
                              stream);
}

// One launch over `n_shards` packed item tables (1: the plain entry points; > 1: hsk_eval_topk_tc_shards, pair kernel only).
static int eval_tc_launch(const void* Uq, int n_shards, const void* const* Vq, const int64_t* rows, const float* const* Ib, int kpad,
                          int precision, const float* Ub, const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be,
                          int64_t n_users, int64_t id_offset, int64_t id_stride, const int64_t* excl_indptr,
                          const int32_t* excl_indices, int k, float* top_scores, int32_t* top_ids, void* scratch,
                          int64_t scratch_bytes, int32_t* status, int variant, hsk_stream_t stream) {
    HSK_REQUIRE(variant >= HSK_EVAL_TC_AUTO && variant <= HSK_EVAL_TC_PAIR, "hsk_eval_topk_tc_v: unknown kernel variant %d", variant);
    const bool pair = variant != HSK_EVAL_TC_SINGLE;
    HSK_REQUIRE(n_shards >= 1 && n_shards <= kMaxItemShards && (pair || n_shards == 1), "hsk_eval_topk_tc: 1..%d item shards (pair kernel)", kMaxItemShards);
    HSK_REQUIRE(Uq && Vq && rows && Ib && u_idx && top_scores && top_ids, "hsk_eval_topk_tc: null pointer");
    HSK_REQUIRE(precision == HSK_PREC_TF32 || precision == HSK_PREC_BF16, "hsk_eval_topk_tc: precision must be TF32 or BF16");
    const bool tf32 = precision == HSK_PREC_TF32;
    const int per_kb = tf32 ? 32 : 64;
    HSK_REQUIRE(kpad >= per_kb && kpad % per_kb == 0, "hsk_eval_topk_tc: kpad must be a multiple of %d", per_kb);
    const int num_kb = kpad / per_kb;
    if (num_kb > TC_MAX_KB)
        return set_err(HSK_ERR_UNSUPPORTED, "hsk_eval_topk_tc: embedding_dim too large for the tensor-core mode (kpad=%d)", kpad);
    HSK_REQUIRE((reinterpret_cast<uintptr_t>(Uq) & 15) == 0, "hsk_eval_topk_tc: operands must be 16-byte aligned");
    HSK_REQUIRE(k >= 1 && k <= kMaxK && Be >= 0, "hsk_eval_topk_tc: bad sizes");
    HSK_REQUIRE((excl_indptr == nullptr) == (excl_indices == nullptr), "hsk_eval_topk_tc: exclusion CSR needs both arrays");
    const int bn = pair ? 2 * TC_BN : TC_BN;
    int64_t max_rows = 0;
    int nt = 0;
    EvalTcArgs a;
    memset(&a, 0, sizeof(a));
    for (int q = 0; q < n_shards; ++q) {
        HSK_REQUIRE(Vq[q] && (reinterpret_cast<uintptr_t>(Vq[q]) & 15) == 0 && rows[q] >= 1, "hsk_eval_topk_tc: item table %d missing, misaligned or empty", q);
        nt += (int)((rows[q] + bn - 1) / bn);
        a.shard_tile_end[q] = nt;
        a.shard_rows[q] = rows[q];
        a.shard_Ib[q] = Ib[q];
        if (rows[q] > max_rows) max_rows = rows[q];
    }
    HSK_REQUIRE(id_stride >= 1 && id_offset >= 0 && id_offset + ((n_shards - 1) + (int64_t)n_shards * (max_rows - 1)) * id_stride < 0x7FFFFFFFll,
                "hsk_eval_topk_tc: bad id mapping");
    if (Be == 0) return HSK_OK;
    a.n_shards = n_shards;
    a.Ub = Ub; a.Ib = Ib[0]; a.Gb = Gb; a.u_idx = u_idx; a.u_rows = u_rows; a.excl_indptr = excl_indptr; a.excl_indices = excl_indices;
    a.n_users = n_users; a.n_local = rows[0]; a.id_offset = id_offset; a.id_stride = id_stride;
    a.Be = Be; a.k = k; a.num_kb = num_kb; a.kelems_per_kb = per_kb;
    tc_plan_tiles(Be, nt, pair, &a.n_tiles, &a.tiles_per_split, &a.n_splits);
    const int64_t need = (int64_t)a.n_splits * Be * TC_CAP * (int64_t)sizeof(uint64_t);
    HSK_REQUIRE(scratch && scratch_bytes >= need, "hsk_eval_topk_tc: scratch too small (%lld < %lld bytes)", (long long)scratch_bytes, (long long)need);
    a.cand = reinterpret_cast<uint64_t*>(scratch);
    a.out_scores = top_scores; a.out_ids = top_ids; a.status = status;
    CUtensorMap tmA;
    EvalTcMaps tmB;
    memset(&tmB, 0, sizeof(tmB));
    int rc = make_map(&tmA, Uq, tf32, kpad, Be, per_kb);
    if (rc) return rc;
    for (int q = 0; q < n_shards; ++q) {
        rc = make_map(&tmB.m[q], Vq[q], tf32, kpad, rows[q], per_kb);
        if (rc) return rc;
    }
    int n_stages = (200 * 1024 - num_kb * TC_TILE_BYTES) / TC_TILE_BYTES;   // ~200 KB of the 227 KB for operands
    if (n_stages > TC_MAX_STAGES) n_stages = TC_MAX_STAGES;
    if (n_stages < 2) n_stages = 2;
    a.n_stages = n_stages;
    const size_t smem = (size_t)(num_kb + n_stages) * TC_TILE_BYTES + 1024;
    cudaStream_t s = as_stream(stream);
    dim3 grid((Be + TC_BM - 1) / TC_BM, a.n_splits);
    cudaError_t e;
    if (pair) {
        rc = launch_eval_tc2(tf32, (int)grid.x, a.n_splits, smem, s, tmA, tmB, a);
        if (rc) return rc;
        e = cudaSuccess;
    } else if (tf32) {
        e = cudaFuncSetAttribute(eval_topk_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) eval_topk_tc_kernel<true><<<grid, TC_THREADS, smem, s>>>(tmA, tmB.m[0], a);
    } else {
        e = cudaFuncSetAttribute(eval_topk_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) eval_topk_tc_kernel<false><<<grid, TC_THREADS, smem, s>>>(tmA, tmB.m[0], a);
    }
    if (e != cudaSuccess) return set_err(HSK_ERR_CUDA, "hsk_eval_topk_tc: smem attribute: %s", cudaGetErrorString(e));
    rc = check_launch("hsk_eval_topk_tc");
    if (rc) return rc;
    if (a.n_splits > 1) rc = launch_merge_keys(a.cand, a.n_splits, Be, TC_CAP, k, top_scores, top_ids, s, Ub, Gb, u_rows ? u_rows : u_idx, u_rows ? (int64_t)1 << 62 : n_users);
    return rc;
}

extern "C" int hsk_eval_topk_tc_v(const void* Uq, const void* Vq, int kpad, int precision, const float* Ub, const float* Ib,
                                  const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be, int64_t n_users,
                                  int64_t n_local, int64_t id_offset, int64_t id_stride, const int64_t* excl_indptr,
                                  const int32_t* excl_indices, int k, float* top_scores, int32_t* top_ids, void* scratch,
                                  int64_t scratch_bytes, int32_t* status, int variant, hsk_stream_t stream) {
    HSK_REQUIRE(Vq && n_local >= 1, "hsk_eval_topk_tc: null pointer / empty item table");
    return eval_tc_launch(Uq, 1, &Vq, &n_local, &Ib, kpad, precision, Ub, Gb, u_idx, u_rows, Be, n_users, id_offset, id_stride,
                          excl_indptr, excl_indices, k, top_scores, top_ids, scratch, scratch_bytes, status, variant, stream);
}

extern "C" int64_t hsk_eval_topk_tc_shards_scratch_bytes(int Be, const int64_t* shard_rows, int n_shards, int k) {
    (void)k;
    if (!shard_rows || n_shards < 1) return 0;
    int nt = 0;
    for (int q = 0; q < n_shards; ++q) nt += (int)((shard_rows[q] + 2 * TC_BN - 1) / (2 * TC_BN));
    int n_tiles, tps, ns;
    tc_plan_tiles(Be > 0 ? Be : 1, nt > 0 ? nt : 1, true, &n_tiles, &tps, &ns);
    return (int64_t)ns * (Be > 0 ? Be : 1) * TC_CAP * (int64_t)sizeof(uint64_t);
}

extern "C" int hsk_eval_topk_tc_shards(const void* Uq, const void* const* Vq_shards, const int64_t* shard_rows,
                                       const float* const* Ib_shards, int n_shards, int kpad, int precision, const float* Ub,
                                       const float* Gb, const int64_t* u_idx, const int64_t* u_rows, int Be, int64_t n_users,
                                       const int64_t* excl_indptr, const int32_t* excl_indices, int k, float* top_scores,
                                       int32_t* top_ids, void* scratch, int64_t scratch_bytes, int32_t* status, hsk_stream_t stream) {
    const float* no_bias[kMaxItemShards] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    return eval_tc_launch(Uq, n_shards, Vq_shards, shard_rows, Ib_shards ? Ib_shards : no_bias, kpad, precision, Ub, Gb, u_idx, u_rows, Be,
                          n_users, 0, 1, excl_indptr, excl_indices, k, top_scores, top_ids, scratch, scratch_bytes, status,
                          HSK_EVAL_TC_PAIR, stream);
}
