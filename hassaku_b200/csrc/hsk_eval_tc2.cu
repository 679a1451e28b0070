// Full-rank evaluator, tensor-core mode, CTA-PAIR kernel: tcgen05.mma.cta_group::2 (UMMA M = 256 over two SMs, N = 256).
//
// Why pairs (measured on the one-CTA kernel, hsk_eval_tc.cu, at 18 944 users x 1 M items x 256, bf16): every CTA streamed
// the whole 512 MB item table through its own shared memory — 75.8 GB of L2 -> SM traffic per batch, 6.9 TB/s, close to
// what the L2 can deliver — and an M128 x N128 MMA reads 8 KB of operands from shared memory per 64 tensor-pipe cycles
// (128 B / clk, the shared-memory port's limit).  A pair shares the item tile: each CTA loads HALF of a 256-item tile
// (128 rows) and the MMA reads both halves through the pair's datapath, so the L2 -> SM traffic and the shared-memory
// bytes per MMA cycle halve; the epilogue's fixed per-tile work (barriers, flags, bias) is amortised over 256 columns.
//
// Per CTA (320 threads, one per SM, clusters of 2 along x; CTA rank 0 = leader):
//   warp 0      TMA producer (both CTAs): its 128-user A tile once (resident), its 128-row half of every item tile through a
//               ring of 16 KB stages (cp.async.bulk.tensor.2d.cta_group::2: the bytes complete on the LEADER's mbarrier)
//   warp 1      leader only: tcgen05.mma.cta_group::2.kind::f16 | tf32, accumulators in BOTH CTAs' TMEM (2 stages x 256 fp32
//               columns = all 512 columns), tcgen05.commit multicast to both CTAs' barriers
//   warps 2-9   epilogue: thread = accumulator lane (user row) x one 128-column half, 4 chunks of 32 columns per tile:
//               tcgen05.ld, a 3-input max tree (16 FMNMX3 per 32 scores) against the row's running k-th score — the item bias
//               is already IN the accumulator: after a stage is read the same warps write the bias row of tile t + 2 into it
//               (tcgen05.st), and the MMA of that tile accumulates on top, so the hot loop has no bias add (FADD per score in
//               the one-CTA kernel) and no shared-memory bias tile; survivors go to the row's candidate list exactly as in
//               hsk_eval_tc.cu (same scan / cut / final-sort code, hsk_eval_tc.cuh).
#include "hsk_eval_tc.cuh"

namespace hsk {

constexpr int T2_BN = 256;                   // items per tile (UMMA_N); each CTA of the pair loads TC_BN = 128 rows of it
constexpr int T2_ACC_STAGES = 2;             // 2 x 256 fp32 columns
// NCG = column groups per tile = epilogue warps / 4 (a warp reads the TMEM lane quarter warp % 4, so the warps that share a
// lane quarter split the tile's columns): NCG = 2 -> 8 epilogue warps x 128 columns, NCG = 4 -> 16 warps x 64 columns.
// A row's 512-entry candidate list has one region per column group; a tile appends at most COLS keys to a region, so a
// region is cut when it holds more than RCAP - COLS, and an intermediate cut keeps <= NCG * (RCAP - COLS) = 256 entries.
// Position of a walk over the launch's tiles in the item shards: the shard's limits live in registers and are re-read from the
// argument block only when the walk crosses into the next shard (once per shard, not once per tile).
struct ShardWalk {
    int gt, q, tile_end;      // global tile, its shard, first tile of the next shard
    int n0, rows;             // first row of the tile inside the shard, rows of the shard (ids fit 31 bits)
    const float* ib;          // the shard's item bias (null: none)
};
__device__ __forceinline__ void walk_load(const EvalTcArgs& a, ShardWalk& w) {
    w.tile_end = a.shard_tile_end[w.q];
    w.rows = (int)a.shard_rows[w.q];
    w.ib = a.shard_Ib[w.q];
}
__device__ __forceinline__ void walk_init(const EvalTcArgs& a, ShardWalk& w, int gt) {
    w.gt = gt;
    w.q = 0;
    while (w.q + 1 < a.n_shards && gt >= a.shard_tile_end[w.q]) ++w.q;
    w.n0 = (gt - (w.q ? a.shard_tile_end[w.q - 1] : 0)) * T2_BN;
    walk_load(a, w);
}
__device__ __forceinline__ void walk_next(const EvalTcArgs& a, ShardWalk& w) {
    ++w.gt;
    w.n0 += T2_BN;
    if (w.gt >= w.tile_end && w.q + 1 < a.n_shards) {
        ++w.q;
        w.n0 = 0;
        walk_load(a, w);
    }
}

#ifndef HSK_T2_SCHED_NUM
#define HSK_T2_SCHED_NUM 3     // schedule ratio 3 / 2 (measurement builds override: profiles/r02_eval_tc2_stall_analysis.md)
#define HSK_T2_SCHED_DEN 2
#endif
template <int NCG> struct T2Cfg {
    static constexpr int WARPS = 4 * NCG;
    static constexpr int THREADS = 64 + WARPS * 32;
    static constexpr int COLS = T2_BN / NCG;
    static constexpr int RCAP = TC_CAP / NCG;
    static constexpr int PRUNE_AT = RCAP - COLS;
    static constexpr int KEEP_MID = NCG * PRUNE_AT;
#ifdef HSK_T2_TRIG
    static constexpr int TRIG = HSK_T2_TRIG;         // measurement builds: cut trigger A/B
#else
    static constexpr int TRIG = PRUNE_AT;
#endif
    static constexpr int GROUP = NCG * 32;           // threads that share a lane quarter
    static constexpr int ROWS_PER_WARP = 32 / NCG;   // rows a warp cuts / finalises
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// the leader CTA's copy of a shared-memory address of this CTA (pairs: CTA rank = bit 24 of the shared::cluster address)
__device__ __forceinline__ uint32_t leader_addr(const void* p) { return smem_u32(p) & 0xFEFFFFFFu; }

__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
            "r"(smem_u32(dst)), "l"(map), "r"(leader_addr(leader_bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {   // arrives on `bar` in BOTH CTAs when the MMAs issued so far retire
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::
                     "r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}
// Arrive on the LEADER CTA's barrier.  No .release.cluster here: that form compiles to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR per
// tile and warp (17 % of the kernel's stall samples, ncu r02); nothing in generic memory is handed over through this
// barrier — the TMEM writes it guards are ordered by tcgen05.wait::st + tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(leader_addr(bar)) : "memory");
}
template <bool TF32>
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_c, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (TF32) {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}\n" ::
                         "r"(tmem_c), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                     : "memory");
    } else {
        asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n" ::
                         "r"(tmem_c), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
                     : "memory");
    }
}
template <bool TF32, int NCG>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(T2Cfg<NCG>::THREADS, 1)
eval_topk_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ EvalTcMaps tmBs, EvalTcArgs a) {
    using Cfg = T2Cfg<NCG>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ uint64_t bar_full[TC_MAX_STAGES], bar_empty[TC_MAX_STAGES], bar_a, bar_tfull[T2_ACC_STAGES], bar_tempty[T2_ACC_STAGES];
    __shared__ uint32_t s_tmem_base;
    __shared__ float s_tau[TC_BM];
    __shared__ uint64_t s_taukey[TC_BM];
    __shared__ int s_cnt[NCG][TC_BM];
    __shared__ int64_t s_exlo[TC_BM], s_exhi[TC_BM];
    __shared__ float s_base[TC_BM];
    __shared__ int s_rowok[TC_BM];
    __shared__ int s_need[4][NCG][2];
    __shared__ __align__(16) float s_ib[4][2][T2_BN];   // per lane quarter: item-bias tiles staged one tile ahead of their TMEM write

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t cta = cluster_ctarank();
    const bool leader = cta == 0;
    const int m0 = blockIdx.x * TC_BM;
    const int split = blockIdx.y;
    const int t_begin = split * a.tiles_per_split;
    const int t_end = min(a.n_tiles, t_begin + a.tiles_per_split);
    const int n_my_tiles = t_end - t_begin;

    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* smA = smem;                                        // num_kb x 16 KB, resident: this CTA's 128 users
    unsigned char* smB = smem + (size_t)a.num_kb * TC_TILE_BYTES;     // n_stages x 16 KB: this CTA's 128 rows of the item tile

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.n_stages; ++s) { mbar_init(&bar_full[s], 1); mbar_init(&bar_empty[s], 1); }
        mbar_init(&bar_a, 1);
        for (int s = 0; s < T2_ACC_STAGES; ++s) { mbar_init(&bar_tfull[s], 1); mbar_init(&bar_tempty[s], 2 * Cfg::WARPS); }
        mbar_fence_init();
    }
    if (warp == 1) {   // TMEM of the pair: the same 512 columns in both CTAs
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&s_tmem_base)), "n"(T2_ACC_STAGES * T2_BN));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n" ::);
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
#pragma unroll
        for (int q = 0; q < NCG; ++q) s_cnt[q][r] = 0;
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();     // both CTAs' barriers are initialised and TMEM allocated before anyone signals across the pair
    tc_fence_after();
    const uint32_t tmem_base = s_tmem_base;

    if (warp == 0) {
        // ===== TMA producer (both CTAs) =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA));
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmBs.m[0]));
            if (leader) mbar_expect_tx(&bar_a, 2u * (uint32_t)a.num_kb * TC_TILE_BYTES);
            for (int kb = 0; kb < a.num_kb; ++kb) tma_load_2d_pair(smA + (size_t)kb * TC_TILE_BYTES, &tmA, kb * a.kelems_per_kb, m0, &bar_a);
            int s = 0;
            uint32_t ph = 0;
            ShardWalk w;
            walk_init(a, w, t_begin);
            for (int t = 0; t < n_my_tiles; ++t) {
                const int n0 = w.n0 + (int)cta * TC_BN;      // this CTA's half of the tile (rows of shard w.q)
                const CUtensorMap* map = &tmBs.m[w.q];
                for (int kb = 0; kb < a.num_kb; ++kb) {
                    mbar_wait(&bar_empty[s], ph ^ 1u);
                    if (leader) mbar_expect_tx(&bar_full[s], 2u * TC_TILE_BYTES);
                    tma_load_2d_pair(smB + (size_t)s * TC_TILE_BYTES, map, kb * a.kelems_per_kb, n0, &bar_full[s]);
                    if (++s == a.n_stages) { s = 0; ph ^= 1u; }
                }
                walk_next(a, w);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA only) =====
        if (leader && lane == 0) {
            // instruction descriptor: D = F32, A = B = BF16 (1) | TF32 (2), K-major both, N = 256, M = 256 (pair)
            const uint32_t fmt = TF32 ? 2u : 1u;
            const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(T2_BN >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
            mbar_wait(&bar_a, 0);
            tc_fence_after();
            int s = 0;
            uint32_t ph = 0;
            for (int t = 0; t < n_my_tiles; ++t) {
                const int as = t & 1;
                mbar_wait(&bar_tempty[as], ((uint32_t)t >> 1) & 1u);   // the epilogues of BOTH CTAs wrote the bias row into this stage
                tc_fence_after();
                const uint32_t tmem_c = tmem_base + (uint32_t)as * T2_BN;
                for (int kb = 0; kb < a.num_kb; ++kb) {
                    mbar_wait(&bar_full[s], ph);
                    tc_fence_after();
                    const uint64_t da = umma_desc(smem_u32(smA + (size_t)kb * TC_TILE_BYTES));
                    const uint64_t db = umma_desc(smem_u32(smB + (size_t)s * TC_TILE_BYTES));
#pragma unroll
                    for (int k = 0; k < TC_KB_BYTES / 32; ++k)   // accumulate = 1 always: the stage holds the bias row
                        tc_mma_pair<TF32>(tmem_c, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, 1u);
                    tc_commit_pair(&bar_empty[s]);
                    if (++s == a.n_stages) { s = 0; ph ^= 1u; }
                }
                tc_commit_pair(&bar_tfull[as]);
            }
        }
    } else {
        // ===== epilogue warps: TMEM lane quarter = warp % 4, column group = (warp - 2) / 4 =====
        const int ew = warp - 2;
        const int quarter = warp & 3;
        const int cg = ew >> 2;
        const int r = quarter * 32 + lane;
        const bool row_ok = s_rowok[r] != 0;
        uint64_t* list = a.cand + ((int64_t)split * a.Be + min(m0 + r, a.Be - 1)) * TC_CAP;
        uint64_t* region = list + cg * Cfg::RCAP;
        int cnt = 0;
        const int bar_id = 1 + quarter;
        const uint32_t tlane = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(cg * Cfg::COLS);
        float* ib_grp = &s_ib[quarter][0][0];
        const int sc0 = cg * Cfg::COLS + lane;   // a warp stages the bias values of ITS columns: sc0 + 32 h, h < STG
        constexpr int STG = T2_BN / Cfg::GROUP;   // bias values a thread stages per tile
        ExCursor ex;
        ex_init(ex, a.excl_indices, s_exlo[r], s_exhi[r]);
        // two walks over this CTA's tiles: `cur` = the tile being scanned, `la` = the tile whose bias row is fetched next (the
        // prologue fetches tiles 0, 1, 2, iteration t fetches tile t + 3: always the next one)
        ShardWalk cur, la;
        walk_init(a, cur, t_begin);
        la = cur;
        int la_tt = 0;        // tile (relative to t_begin) `la` stands on
        auto ib_la = [&](int col) -> float {    // bias of column `col` of the tile `la` stands on (0 beyond the shard / the CTA's range)
            return (la.ib && la_tt < n_my_tiles && la.n0 + col < la.rows) ? __ldg(la.ib + la.n0 + col) : 0.f;
        };
        auto la_next = [&]() { walk_next(a, la); ++la_tt; };
        int cur_q = cur.q;

        // prologue: bias rows of the first two tiles into the stages (through the group's staging tile), stages to the MMA warp
        for (int ts = 0; ts < T2_ACC_STAGES && ts < n_my_tiles; ++ts) {
#pragma unroll
            for (int h = 0; h < STG; ++h) ib_grp[sc0 + 32 * h] = ib_la(sc0 + 32 * h);
            la_next();
            named_bar_sync(bar_id, Cfg::GROUP);
            tc_write_bias<Cfg::COLS / 32>(ib_grp + cg * Cfg::COLS, tlane + (uint32_t)ts * T2_BN);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(&bar_tempty[ts]);
            named_bar_sync(bar_id, Cfg::GROUP);
        }
#pragma unroll
        for (int h = 0; h < STG; ++h) ib_grp[sc0 + 32 * h] = ib_la(sc0 + 32 * h);   // slot 0 <- tile 2
        la_next();
        named_bar_sync(bar_id, Cfg::GROUP);

        int next_cut = 2;          // tiles after which every row is cut: 2, 3, 4, 6, 9, 13, ... (ratio HSK_T2_SCHED_NUM / DEN)
        for (int t = 0; t < n_my_tiles; ++t) {
            const int as = t & 1;
            const int q = cur.q;
            const int n0 = cur.n0;
            if (q != cur_q) {      // the next shard's item ids start low again: rewind the exclusion cursor
                cur_q = q;
                ex_init(ex, a.excl_indices, s_exlo[r], s_exhi[r]);
            }
            const int ncols = min(T2_BN, cur.rows - n0);
            walk_next(a, cur);     // (q, n0, ncols of THIS tile are latched above)
            // item id of (shard q, row n) = id_offset + (q + n_shards * n) * id_stride
            const uint32_t id_step = (uint32_t)(a.n_shards * a.id_stride);
            const uint32_t id_base = (uint32_t)a.id_offset + ((uint32_t)q + (uint32_t)a.n_shards * (uint32_t)n0) * (uint32_t)a.id_stride;
            const float tau = s_tau[r];
            const uint64_t taukey = s_taukey[r];
            // the bias values the NEXT iteration writes (tile t + 3): in flight during this tile
            float ibn[STG];
#pragma unroll
            for (int h = 0; h < STG; ++h) ibn[h] = ib_la(sc0 + 32 * h);
            la_next();
            mbar_wait(&bar_tfull[as], ((uint32_t)t >> 1) & 1u);
            tc_fence_after();
            const uint32_t taddr = tlane + (uint32_t)as * T2_BN;
#pragma unroll 1
            for (int cp = 0; cp < Cfg::COLS / 64; ++cp) {       // two 32-column chunks at a time: 64 accumulator registers live
                uint32_t raw0[32], raw1[32];
                tc_ld32_issue(taddr + (uint32_t)(cp * 64), raw0);
                tc_ld32_issue(taddr + (uint32_t)(cp * 64 + 32), raw1);
                tc_ld_wait();
                auto chunk = [&](const uint32_t (&raw)[32], int cc) {
                    const int c = cg * Cfg::COLS + cp * 64 + cc * 32;     // column of the tile
                    if (c >= ncols) return;
                    float v[32], g[8];
#pragma unroll
                    for (int e = 0; e < 32; ++e) v[e] = __uint_as_float(raw[e]);
                    const float mx = tc_chunk_max(v, g);
#ifdef HSK_MEASURE_NOSCAN   // measurement builds only (never the shipped library): the epilogue without its candidate scan
                           // after the first 4 tiles -> 6.39 ms = 1 517 TFLOP/s at 18 944 x 1 M x 256 (shipped: 9.95 ms)
                    if (row_ok && mx >= tau && t < 4)
#else
                    if (row_ok && mx >= tau)
#endif
                        tc_scan_groups(v, g, tau, taukey, id_base + (uint32_t)c * id_step, id_step, cnt, region, ex, ncols - c);
                };
                chunk(raw0, 0);
                chunk(raw1, 1);
            }
            // the stage has been read: write the bias row of tile t + 2 into it and hand it back to the MMA warp
            if (t + T2_ACC_STAGES < n_my_tiles) {
                tc_write_bias<Cfg::COLS / 32>(ib_grp + (t & 1) * T2_BN + cg * Cfg::COLS, taddr);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(&bar_tempty[as]);
            }
#pragma unroll
            for (int h = 0; h < STG; ++h) ib_grp[((t + 1) & 1) * T2_BN + sc0 + 32 * h] = ibn[h];   // staging slot of tile t + 3
            const bool last = (t + 1 == n_my_tiles);
            // scheduled cut: EVERY row of the CTA pair is cut after the same tiles, a geometric schedule (the k-th best score of a
            // random stream needs ~k new candidates per doubling of the items seen).  Cuts triggered by a region filling up
            // hit a different row in nearly every tile and each one stalled the warp pair, then the accumulator stage, then
            // the MMA and the other CTA for ~1.5 k cycles; now the stall is paid ~20 times per launch by all warps at once and
            // the fill trigger only fires for rows whose scores do not arrive in random order.
            bool sched = false;
            if (t + 1 == next_cut) {
                sched = true;
                const int step = (next_cut * (HSK_T2_SCHED_NUM - HSK_T2_SCHED_DEN)) / HSK_T2_SCHED_DEN;
                next_cut += step > 1 ? step : 1;
            }
#ifdef HSK_MEASURE_NOPAIRBAR   // measurement builds only: no fill trigger, so no per-tile barrier of the two warps (UNSAFE for sorted streams)
            __syncwarp();
            int grp_need = (last || sched) ? 1 : 0;
#else
            const bool warp_need = __any_sync(kFull, row_ok && cnt > Cfg::TRIG) || last || sched;
            if (lane == 0) s_need[quarter][cg][t & 1] = warp_need ? 1 : 0;
            named_bar_sync(bar_id, Cfg::GROUP);
            int grp_need = 0;
#pragma unroll
            for (int q = 0; q < NCG; ++q) grp_need |= s_need[quarter][q][t & 1];
#endif
            if (grp_need) {
                s_cnt[cg][r] = cnt;
                named_bar_sync(bar_id, Cfg::GROUP);
                int my_c[NCG];
                bool my_need = false;
#pragma unroll
                for (int q = 0; q < NCG; ++q) my_c[q] = 0;
                if (lane < Cfg::ROWS_PER_WARP) {   // lane j looks at row j of this warp's rows
                    const int rj = quarter * 32 + cg * Cfg::ROWS_PER_WARP + lane;
                    my_need = last || sched;
#pragma unroll
                    for (int q = 0; q < NCG; ++q) { my_c[q] = s_cnt[q][rj]; my_need |= my_c[q] > Cfg::TRIG; }
                    my_need = my_need && s_rowok[rj];
                }
                unsigned need = __ballot_sync(kFull, my_need);
                while (need) {
                    const int j = __ffs(need) - 1;
                    need &= need - 1;
                    const int rr = quarter * 32 + cg * Cfg::ROWS_PER_WARP + j;
                    int cc[NCG];
#pragma unroll
                    for (int q = 0; q < NCG; ++q) cc[q] = __shfl_sync(kFull, my_c[q], j);
                    uint64_t* lp = a.cand + ((int64_t)split * a.Be + (m0 + rr)) * TC_CAP;
                    float ntau;
                    uint64_t ntaukey;
                    // intermediate cuts keep <= KEEP_MID entries (<= PRUNE_AT per region, so the next tile's appends cannot
                    // overflow a region); the last cut keeps <= 192 in all for the final sort
                    const int total = tc_cut_row<NCG>(lp, cc, a.k, lane, last ? 192 : Cfg::KEEP_MID, &ntau, &ntaukey);
                    __syncwarp();
                    if (lane == 0) {
#pragma unroll
                        for (int q = 0; q < NCG; ++q) s_cnt[q][rr] = (total - q + NCG - 1) / NCG;
                        s_tau[rr] = ntau; s_taukey[rr] = ntaukey;
                    }
                    if (last) {
                        int n_final = total;
                        if (total < a.k) {
                            // this split's tiles [t_begin, t_end): id = id_offset + (q + n_shards * n) * id_stride for row n of
                            // shard q, in global tile shard_tile_end[q - 1] + n / T2_BN
                            const bool one = a.n_shards == 1;
                            const int64_t n_hi = one ? min((int64_t)t_end * T2_BN, a.shard_rows[0]) - 1 : 0;
                            n_final = tc_fill_excluded<NCG>(lp, total, a.k, lane, a.excl_indices, s_exlo[rr], s_exhi[rr],
                                                            (uint32_t)(a.id_offset + (one ? (int64_t)t_begin * T2_BN * a.id_stride : 0)),
                                                            one ? (uint32_t)(a.id_offset + n_hi * a.id_stride) : 0xFFFFFFFFu,
                                                            [&](uint32_t id) {
                                const int64_t rel = (int64_t)id - a.id_offset;
                                if (rel < 0 || rel % a.id_stride != 0) return false;
                                const int64_t j = rel / a.id_stride;
                                const int qq = (int)(j % a.n_shards);
                                const int64_t n = j / a.n_shards;
                                if (n >= a.shard_rows[qq]) return false;
                                const int64_t gt = (qq ? a.shard_tile_end[qq - 1] : 0) + n / T2_BN;
                                return gt >= t_begin && gt < t_end;
                            });
                        }
                        uint64_t keys[kKeysPerLane];
                        tc_final_sort<NCG>(lp, n_final, a.k, lane, keys);
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
                named_bar_sync(bar_id, Cfg::GROUP);
                cnt = s_cnt[cg][r];
            }
        }
        // rows with a bad user index: empty lists / -1 ids
        for (int j = 0; j < Cfg::ROWS_PER_WARP; ++j) {
            const int rr = quarter * 32 + cg * Cfg::ROWS_PER_WARP + j;
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

    // neither CTA may leave (or free its TMEM) while its peer can still read its shared memory or signal its barriers
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(T2_ACC_STAGES * T2_BN));
    }
}

template <bool TF32, int NCG>
static int launch_tc2(dim3 grid, size_t smem, cudaStream_t s, const CUtensorMap& tmA, const EvalTcMaps& tmB, const EvalTcArgs& a) {
    cudaError_t e = cudaFuncSetAttribute(eval_topk_tc2_kernel<TF32, NCG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_err(HSK_ERR_CUDA, "hsk_eval_topk_tc(pair): smem attribute: %s", cudaGetErrorString(e));
    eval_topk_tc2_kernel<TF32, NCG><<<grid, T2Cfg<NCG>::THREADS, smem, s>>>(tmA, tmB, a);
    return check_launch("hsk_eval_topk_tc(pair)");
}

// launcher (called by hsk_eval_topk_tc_v in hsk_eval_tc.cu): grid.x = an even number of 128-user tiles.
// NCG = 2 (8 epilogue warps x 128 columns) is the only shipped instantiation: NCG = 4 (16 warps x 64 columns, 96 registers,
// four list regions per row) was measured at 10.69 ms against 9.96 ms for NCG = 2 (18 944 x 1 M x 256, bf16) — the
// epilogue is not bound by a single warp's instruction latency but by the candidate scan itself (see HSK_MEASURE_NOSCAN).
int launch_eval_tc2(bool tf32, int row_tiles, int n_splits, size_t smem, cudaStream_t s, const CUtensorMap& tmA,
                    const EvalTcMaps& tmB, const EvalTcArgs& a) {
    dim3 grid((unsigned)((row_tiles + 1) / 2 * 2), (unsigned)n_splits);
    return tf32 ? launch_tc2<true, 2>(grid, smem, s, tmA, tmB, a) : launch_tc2<false, 2>(grid, smem, s, tmA, tmB, a);
}

}  // namespace hsk
