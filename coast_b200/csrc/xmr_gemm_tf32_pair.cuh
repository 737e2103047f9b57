// xmr_gemm_tf32_pair.cuh -- the protected TF32 matmul of xmr_gemm_tf32.cuh on CTA PAIRS (tcgen05 cta_group::2).
//
// Why: the chip's L2 delivers ~6300 B/clk to all SMs together (B300_MICROARCH.md "LTS throughput cap") = 42.6 B/clk/SM.  A
// single-CTA 128 x 256 tile streams 48 KiB of operands per 512 tensor cycles = 96 B/clk/SM at full rate, a 128 x 128 DWC tile
// 64 B/clk/SM, the TMR tile 42.7 B/clk/SM: the unprotected and DWC kernels are L2->SM bound, the TMR kernel sits on the edge.
// Two CTAs of one TPC (cluster 2 x 1 x 1) that share a 256 x BN tile each stage only HALF of the B tile; the pair's MMA
// (M = 256, issued by the leader CTA) reads A from both CTAs' shared memory and the two B halves from either side:
//     unprotected  256 x 256 pair tile : 32 KiB per CTA per 512 cycles = 64 B/clk/SM   (was 96), two accumulator sets
//     DWC          256 x 128           : 24 KiB per 512 cycles         = 48 B/clk/SM   (was 64), two accumulator sets (2 x 2 x 128 = 512
//                                        TMEM columns): the epilogue of tile i overlaps the main loop of tile i+1
//     TMR          256 x 128           : 24 KiB per 768 cycles         = 32 B/clk/SM   (was 42.7); one accumulator set as before
// Measured (B200, 4096^3): the TMR kernel does not move (0.465 vs 0.463 ms: tensor-pipe bound), so TMR always runs the single-CTA kernel.
// Everything else is the single-CTA kernel: NC accumulators per CTA in TMEM (each CTA holds its own 128 rows x BN columns x NC),
// the same voting epilogue (epilogue_cols), the same counters and fault site, the same per-element accumulation order over K --
// outputs are bit-identical to xmr_gemm_tf32_* (tests/test_gpu_gemm.py).
//
// Protocol (s = stage):
//   full[s]        lives in the LEADER's shared memory (count 1): the leader's producer arms it with the bytes of BOTH CTAs; the
//                  peer's TMA completes its transactions on it remotely (cp.async.bulk.tensor ... .cta_group::2);
//   empty[s]       one per CTA; the MMA's commit multicasts the arrive to both (tcgen05.commit ... multicast::cluster, mask 0b11);
//   tmem_full[b]   one per CTA, same multicast commit;
//   tmem_empty[b]  in the LEADER (count 2 x 8 warps): every epilogue warp of both CTAs arrives once per tile (the peer's remotely).
// Warp roles per CTA as in the single-CTA kernel (TMA producer / MMA issuer (leader CTA only) / TMEM allocator / 8 epilogue warps).
#pragma once
#include "xmr_gemm_tf32.cuh"

namespace xmr {
namespace gemm {

template <int NC> struct PairGeom {
    static constexpr int BN = NC == 1 ? 256 : 128;               // pair tile = 256 x BN
    static constexpr int BNH = BN / 2;                           // B columns each CTA stages
    static constexpr int ACC_BUFS = NC == 3 ? 1 : 2;             // 1 x 256 x 2, 2 x 128 x 2 = 512 columns; 3 x 128 leaves no second set
    static constexpr int STAGES = NC == 1 ? 6 : 8;               // 32 KiB / 24 KiB per stage: 192 KiB either way
    static constexpr uint32_t B_STAGE = BK * BNH * 4;
    static constexpr uint32_t ACC_COLS = (uint32_t)NC * BN * ACC_BUFS;
    static_assert(ACC_COLS <= TMEM_COLS, "TMEM budget");
    static constexpr uint32_t SMEM_BYTES = STAGES * (A_STAGE + B_STAGE) + 1024 + 256;
    // as Geom::IDESC with M = 256 (the pair), N = BN
    static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
};

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_smem_addr` in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank)); return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads of a CTA pair: the bytes land in THIS CTA's shared memory, the transaction completes on the barrier at `bar_cluster`
// (a shared::cluster address: the leader's full[s])
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma2_load_3d(void* smem_dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "l"(pol) : "memory");
}
template <int USAGE>                                            // A-operand collector usage, as tc_mma_tf32_col
__device__ __forceinline__ void tc2_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if (USAGE == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 2)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32.collector::a::use [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 3)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once all previously issued MMAs have retired
__device__ __forceinline__ void tc2_commit_both(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// mbarrier wait that cannot hang the GPU: a pair protocol error (a lost remote arrival) traps after ~2^26 polls instead of spinning
__device__ __forceinline__ void mbar_wait_or_trap(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    for (uint32_t spins = 0; spins < (1u << 26); ++spins) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
    }
    asm volatile("trap;");
}

template <int NC, bool INJECT>
__device__ __forceinline__ void gemm_pair_body(const xmr_args& a, const CUtensorMap* map_a, const CUtensorMap* map_b) {
    using G = PairGeom<NC>;
    constexpr int BN = G::BN, STAGES = G::STAGES, ACC_BUFS = G::ACC_BUFS;
    constexpr uint32_t B_STAGE = G::B_STAGE;
    extern __shared__ uint8_t smem_dyn[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023u) & ~(uintptr_t)1023u);
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (A_STAGE + B_STAGE));
    uint64_t* full = bars;                                      // [STAGES]   used in the leader only
    uint64_t* empty = bars + STAGES;                            // [STAGES]   per CTA
    uint64_t* tmem_full = bars + 2 * STAGES;                    // [ACC_BUFS] per CTA
    uint64_t* tmem_empty = bars + 2 * STAGES + ACC_BUFS;        // [ACC_BUFS] used in the leader only
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 2 * ACC_BUFS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                    // 0 = leader (issues the MMAs), 1 = peer
    const uint32_t pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const uint32_t tiles_n = a.N / BN, tiles_m = a.M / 256u, n_tiles = tiles_m * tiles_n, kblocks = a.K / BK;
    // rasterisation in units of 256-row pair tiles: half as many tile-rows per group as the single-CTA kernel's 128-row tiles
    constexpr uint32_t group_m = GROUP_M / 2u;
    // short last round (unprotected kernel): its tiles run as two 256 x 128 halves, as in the single-CTA kernel (`decode` there)
    uint32_t sched_full = n_tiles, n_virtual = n_tiles;
    if (NC == 1) {
        const uint32_t whole = (n_tiles / n_pairs) * n_pairs, rem = n_tiles - whole;
        if (rem && 2u * rem <= n_pairs) { sched_full = whole; n_virtual = whole + 2u * rem; }
    }
    auto decode = [&](uint32_t v, uint32_t& tm, uint32_t& n_off, uint32_t& bn_t) {
        uint32_t w = v, h = 0, tn;
        bn_t = BN;
        if (v >= sched_full) { w = sched_full + ((v - sched_full) >> 1); h = (v - sched_full) & 1u; bn_t = BN / 2; }
        tile_coords(w, tiles_m, tiles_n, group_m, tm, tn);
        n_off = tn * BN + h * (BN / 2);
    };

    if (threadIdx.x == 0) {
        tma_prefetch_desc(map_a); tma_prefetch_desc(map_b);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < ACC_BUFS; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], 2 * (EPI_THREADS / 32)); }
        fence_barrier_init();
    }
    if (warp == 2) {                                            // the same warp of BOTH CTAs allocates (and later frees) the pair's TMEM
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                         // the peer's barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer (both CTAs): own 128 rows of A, own half of the B columns; transactions complete on the LEADER's full[s]
        uint32_t it = 0;
        const uint64_t pol_a = l2_policy_evict_last(), pol_b = l2_policy_evict_first();
        for (uint32_t tile = pair; tile < n_virtual; tile += n_pairs) {
            uint32_t tm, n_off, bn_t;
            decode(tile, tm, n_off, bn_t);
            const uint32_t bnh_t = bn_t / 2u;                   // this CTA's share of the tile's B columns
            const int m0 = (int)(tm * 256u + rank * 128u), n0 = (int)(n_off + rank * bnh_t);
            const int b_loads = (int)bnh_t / 64;                // the B box is {32 n, 32 k, 2 chunks} = 64 columns
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                mbar_wait_or_trap(&empty[s], ph ^ 1u);
                if (rank == 0) mbar_arrive_expect_tx(&full[s], 2u * (A_STAGE + bnh_t * BK * 4u));
                const uint32_t bar = mapa_u32(smem_u32(&full[s]), 0);
                tma2_load_2d(sA + s * A_STAGE, map_a, bar, (int)(kb * BK), m0, pol_a);                  // box {32 k, 128 m}
                for (int c = 0; c < b_loads; ++c)
                    tma2_load_3d(sB + s * B_STAGE + c * (2 * BK * 128), map_b, bar, 0, (int)(kb * BK), n0 / 32 + 2 * c, pol_b);
            }
        }
    } else if (warp == 1 && rank == 0) {
        // ===== MMA issuer (leader CTA): M = 256 across the pair, every MMA issued NC times into NC accumulators
        const bool leader = elect_one();
        uint32_t it = 0, tcount = 0;
        for (uint32_t tile = pair; tile < n_virtual; tile += n_pairs, ++tcount) {
            const uint32_t buf = tcount % ACC_BUFS, use = tcount / ACC_BUFS;
            const uint32_t bn_t = tile >= sched_full ? BN / 2 : BN;
            const uint32_t idesc = (G::IDESC & ~(0x3Fu << 17)) | ((bn_t >> 3) << 17);      // MMA N of this tile
            mbar_wait_or_trap(&tmem_empty[buf], (use & 1u) ^ 1u);       // both CTAs' epilogues drained this accumulator set
            tc_fence_after();
            const uint32_t acc0 = tmem_base + buf * (uint32_t)(NC * BN);
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                mbar_wait_or_trap(&full[s], ph);
                tc_fence_after();
                if (leader) {
                    const uint64_t da0 = smem_desc(smem_u32(sA + s * A_STAGE), 16, 1024, SWZ_128B);
                    const uint64_t db0 = smem_desc(smem_u32(sB + s * B_STAGE), BK * 128, 512, SWZ_128B_BASE32B);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t da = da0 + (uint64_t)((k * UMMA_K * 4) >> 4), db = db0 + (uint64_t)((k * 1024) >> 4);
                        const uint32_t acc = (kb | (uint32_t)k) ? 1u : 0u;
                        if (NC == 1) {
                            tc2_mma_tf32<0>(acc0, da, db, idesc, acc);
                        } else {                                // A stays in the collector across the replicas of this k-step
                            tc2_mma_tf32<1>(acc0, da, db, idesc, acc);
                            if (NC == 3) tc2_mma_tf32<2>(acc0 + BN, da, db, idesc, acc);
                            tc2_mma_tf32<3>(acc0 + (NC - 1) * BN, da, db, idesc, acc);
                        }
                    }
                    tc2_commit_both(&empty[s]);                 // both CTAs' slots are free once these MMAs retire
                }
                __syncwarp();
            }
            if (leader) tc2_commit_both(&tmem_full[buf]);       // both CTAs' accumulators are complete
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ===== epilogue (both CTAs): own 128 rows of the pair tile
        const int q = warp & 3, half = (warp - 4) >> 2;
        const uint64_t pol_c = l2_policy_evict_first();
        Tally tally(a);
        uint32_t tcount = 0;
        for (uint32_t tile = pair; tile < n_virtual; tile += n_pairs, ++tcount) {
            uint32_t tm, n0, bn_t;
            decode(tile, tm, n0, bn_t);
            const uint32_t m0 = tm * 256u + rank * 128u;
            const uint32_t buf = tcount % ACC_BUFS, use = tcount / ACC_BUFS;
            mbar_wait_or_trap(&tmem_full[buf], use & 1u);
            tc_fence_after();
            const uint32_t row = m0 + q * 32 + lane;
            const uint32_t lane_addr = tmem_base + buf * (uint32_t)(NC * BN) + ((uint32_t)(q * 32) << 16);
            epilogue_cols<NC, INJECT>(a, tally, lane_addr, (uint32_t)BN, row, n0, half * (int)(bn_t / 2), (half + 1) * (int)(bn_t / 2), pol_c);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty[buf]), 0));     // one arrival per warp, on the leader's barrier
        }
        tally.flush(a.counters);
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                         // nobody leaves (or frees TMEM) while the pair's MMAs / remote arrivals are in flight
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

}  // namespace gemm
}  // namespace xmr

#define XMR_GEMM_PAIR_KERNEL(NC, INJ)                                                                    \
    extern "C" __global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(xmr::gemm::CTA_THREADS, 1)    \
    xmr_gemm_tf32p_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap map_a, \
                                     const __grid_constant__ CUtensorMap map_b) {                        \
        xmr::gemm::gemm_pair_body<NC, INJ != 0>(a, &map_a, &map_b);                                      \
    }
XMR_GEMM_PAIR_KERNEL(1, 0) XMR_GEMM_PAIR_KERNEL(2, 0)
XMR_GEMM_PAIR_KERNEL(1, 1) XMR_GEMM_PAIR_KERNEL(2, 1)
