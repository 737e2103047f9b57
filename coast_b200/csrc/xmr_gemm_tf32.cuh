// xmr_gemm_tf32.cuh -- protected dense matmul on the 5th-gen tensor cores (BASELINE config 4).
//
// C[M,N] = A[M,K] . B[K,N], fp32 in / fp32 out, row-major, tcgen05.mma kind::tf32 (operands are read
// as TF32 = top 19 bits of each fp32; fp32 accumulate in TMEM).  It is the tensor-core realisation of
// matrix_multiply() (tests/matrixMultiply/matrixMultiply.c:95-112, tests/mm_common/mm_common_tmr.c:3-20);
// the bit-exact integer flavour of those loops is xmr_mm.cuh.
//
// Redundancy costs FLOPs, not bandwidth:
//   * ONE copy of each A/B tile is staged in shared memory by TMA (128B swizzle; 32-byte atoms for the
//     N-contiguous B operand), 6-stage mbarrier ring;
//   * the single MMA-issuing thread issues every tcgen05.mma NC times, once per replica, against NC
//     DIFFERENT TMEM accumulators (columns [r*128, r*128+128)) -- the replicas of cloneInsns
//     (cloning.cpp:2189-2204) are NC independent accumulator tiles fed from the same operand bytes;
//   * the epilogue warps read the NC accumulators back (tcgen05.ld), vote element-wise with the reference's
//     select voter and `fcmp oeq` (synchronization.cpp:57-62,512-522), count disagreements
//     (:1391-1431), and write ONE voted C tile.
// Unit = one C element (the `mm_t` store, mm_common_tmr.c:16); local unit index = i*N + j.
// Fault site 0 = the replica's final accumulator value (32 bits) as read back for the vote.
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator,
// warps 4..11 = epilogue (TMEM lane quarter = warp % 4, column half = (warp - 4) / 4).  Persistent CTAs, one per SM.
//
// r02: an SS-mode kind::tf32 MMA of 128 x 128 x 8 reads 8 KiB of operands from shared memory for 64 tensor-pipe cycles =
// 128 B/clk, exactly the SM's shared-memory bandwidth -- the r01 kernels were shared-memory-read bound (ncu: tensor pipe
// 70 % unprotected).  Two remedies, chosen per replica count (Geom<NC>):
//   NC >= 2 : the NC replica MMAs of a k-step keep A in the tensor core's collector (tc_mma_tf32_col): shared-memory reads drop
//             from 128 to 85 (TMR) / 96 (DWC) B/clk.  Staging A in TMEM instead (tcgen05.cp + TS-mode MMAs) reads as little and
//             was measured no faster (B200, 4096^3: TMR 0.498 vs 0.495 ms; DWC 0.354 ms): the replicated MMAs are bound by the
//             tensor pipe itself (830 TF/s issued = 96 % of the measured cuBLAS-derived TF32 peak), not by shared-memory reads.
//   NC == 1 : tile 128 x 256 (MMA N = 256: 12 KiB per 128 cycles = 96 B/clk) with TWO accumulator buffers, so the epilogue
//             of tile i overlaps the main loop of tile i+1.
#pragma once
#include "xmr_common.cuh"

namespace xmr {
namespace gemm {

constexpr int BM = 128, BK = 32;                     // BK fp32 = 128 bytes = one swizzle row
constexpr int UMMA_K = 8;                            // 32 bytes of tf32
constexpr uint32_t A_STAGE = BM * BK * 4;            // 16 KiB
constexpr uint32_t TMEM_COLS = 512;
constexpr int CTA_THREADS = 384, EPI_THREADS = 256;     // warps 0-2 = TMA / MMA / TMEM alloc, warp 3 idle, warps 4-11 = epilogue
template <int NC, bool WIDE = (NC == 1)> struct Geom {         // WIDE: 128 x 256 tiles (unprotected, N % 256 == 0)
    static constexpr int BN = WIDE ? 256 : 128;
    static constexpr int STAGES = WIDE ? 4 : 6;
    static constexpr int ACC_BUFS = NC == 3 ? 1 : 2;             // accumulator sets: double-buffered when TMEM allows (1 x 256 x 2, 2 x 128 x 2 = 512 columns)
    static constexpr uint32_t B_STAGE = BK * BN * 4;              // laid out [BN/32 chunks][BK rows][128 B]
    static constexpr uint32_t ACC_COLS = (uint32_t)NC * BN * ACC_BUFS;
    static_assert(ACC_COLS <= TMEM_COLS, "TMEM budget");
    static constexpr uint32_t SMEM_BYTES = STAGES * (A_STAGE + B_STAGE) + 1024 /*align slack*/ + 256 /*barriers*/;
    // Instruction descriptor: c_format F32 (1) [4,6), a/b_format TF32 (2) [7,10)/[10,13), a_major K (0) [15], b_major MN (1) [16]
    // (B is row-major K x N: N contiguous), N>>3 [17,23), M>>4 [24,29)
    static constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
};
constexpr uint32_t GROUP_M = 16;                     // tile rasterisation: 16 tile-rows per group, column-major inside

// Persistent CTAs take tiles blockIdx.x, +grid, ...; consecutive tile ids therefore run concurrently.  Row-major ids
// make one wave touch ~5 A row-blocks and ALL of B (ncu r01: 489 MB read for 134 MB of operands); grouping 16 tile-rows
// and walking columns inside the group keeps a wave on ~16 A row-blocks x ~10 B column-blocks, which the 126 MB L2 holds.
__device__ __forceinline__ void tile_coords(uint32_t tile, uint32_t tiles_m, uint32_t tiles_n, uint32_t group_m, uint32_t& tm, uint32_t& tn) {
    const uint32_t per_group = group_m * tiles_n;
    const uint32_t g = tile / per_group, w = tile - g * per_group;
    const uint32_t rows = min(group_m, tiles_m - g * group_m);
    tm = g * group_m + w % rows;
    tn = w / rows;
}

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// L2 eviction-priority hints: A loads evict_last, B loads and C stores evict_first, so A stays in the 126 MB L2 while B streams
// through and C is written once (5 % fewer DRAM reads at 4096^3, same time: profiles/r02_gemm_l2_sweep.txt).
__device__ __forceinline__ uint64_t l2_policy_evict_last() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t l2_policy_evict_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_load_3d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_v4_hint(void* p, uint4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {      // arrives on `bar` when all previously issued MMAs retire
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// The replicas of one k-step are NC back-to-back MMAs on the SAME operands.  The A-operand collector of the tensor core can keep A
// across them (collector::a::fill on the first, ::use in between, ::lastuse on the last; SASS UTCHMMA ...A_KEEP / A_REUSE): A is then read
// from shared memory once per k-step instead of NC times (TMR: 16 KiB per 3 MMAs instead of 24 = 85 B/clk instead of 128).
// USAGE: 0 = plain (collector::a::discard, the default), 1 = fill, 2 = use, 3 = lastuse.
template <int USAGE>
__device__ __forceinline__ void tc_mma_tf32_col(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if (USAGE == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 2)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32.collector::a::use [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 3)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else
        tc_mma_tf32(d_tmem, a_desc, b_desc, idesc, accumulate);
}
// 32 lanes x 32 consecutive fp32 columns: thread = TMEM lane (row), registers = columns
__device__ __forceinline__ void tc_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ bool elect_one() {       // one lane of a CONVERGED warp (SASS ELECT)
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor: start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46), fixed 0b001 [46,49),
// swizzle mode [61,64): 2 = SWIZZLE_128B (16-byte atoms), 1 = SWIZZLE_128B_BASE32B (32-byte atoms).
// Bring-up on the B200 (tools/probe/tc_probe.cu): an MN-major TF32 operand is only read correctly with the
// 32-byte-atom swizzle (TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B); with plain SWIZZLE_128B the MMA returns zeros.
constexpr uint32_t SWZ_128B = 2, SWZ_128B_BASE32B = 1;
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t swizzle) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)swizzle << 61);
}
// Epilogue of one accumulator row: columns [c_begin, c_end) of a tile whose replica r lives at TMEM columns lane_addr + r * rep_stride.
// TMEM -> registers, (inject), vote with the reference's select voter / `fcmp oeq`, count, ONE store of the voted row segment.
template <int NC, bool INJECT>
__device__ __forceinline__ void epilogue_cols(const xmr_args& a, Tally& tally, uint32_t lane_addr, uint32_t rep_stride, uint32_t row, uint32_t n0,
                                              int c_begin, int c_end, uint64_t pol_c) {
    const uint32_t flags = a.flags;
    const bool majority = flags & COAST_F_MAJORITY_D;
    float* C = static_cast<float*>(a.out);
#pragma unroll 1
    for (int c0 = c_begin; c0 < c_end; c0 += 32) {
        uint32_t v[3][32];
#pragma unroll
        for (int r = 0; r < NC; ++r) tc_ld_32x32(lane_addr + r * rep_stride + c0, v[r]);
        tc_wait_ld();
        float* dst = C + (size_t)row * a.N + n0 + c0;
        const unsigned long long local0 = (unsigned long long)row * a.N + n0 + c0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                uint32_t r0 = v[0][j + e], r1 = NC > 1 ? v[1][j + e] : r0, r2 = NC > 2 ? v[2][j + e] : r0;
                if (INJECT) {
                    Fault f = fault_for_unit(a, NC, local0 + j + e, [](uint32_t) { return 32u; });
                    if (f.active) {
                        tally.injected++;
                        uint32_t mk = 1u << f.bit;
                        if (f.replica == 0) r0 ^= mk; else if (f.replica == 1) r1 ^= mk; else r2 ^= mk;
                    }
                }
                const float f0 = __uint_as_float(r0), f1 = __uint_as_float(r1), f2 = __uint_as_float(r2);
                uint32_t vote = r0, bad = 0;
                if (NC == 2) bad = (f0 == f1) ? 0u : 1u;
                if (NC == 3) {
                    const bool c01 = (f0 == f1), c02 = (f0 == f2);       // fcmp oeq
                    vote = majority ? ((r0 & r1) | (r0 & r2) | (r1 & r2)) : (c01 ? r0 : r2);
                    bad = (c01 && c02) ? 0u : 1u;
                }
                o[e] = vote;
                tally.unit_exit<NC>(bad, 1u, flags, a.unit_base + local0 + j + e);
            }
            st_v4_hint(dst + j, make_uint4(o[0], o[1], o[2], o[3]), pol_c);
        }
    }
}

template <int NC, bool INJECT, bool WIDE = (NC == 1)>
__device__ __forceinline__ void gemm_body(const xmr_args& a, const CUtensorMap* map_a, const CUtensorMap* map_b) {
    using G = Geom<NC, WIDE>;
    constexpr int BN = G::BN, STAGES = G::STAGES, ACC_BUFS = G::ACC_BUFS;
    constexpr uint32_t B_STAGE = G::B_STAGE;
    extern __shared__ uint8_t smem_dyn[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023u) & ~(uintptr_t)1023u);
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * A_STAGE;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (A_STAGE + B_STAGE));
    uint64_t* full = bars;                 // [STAGES]  TMA -> MMA
    uint64_t* empty = bars + STAGES;       // [STAGES]  MMA -> TMA
    uint64_t* tmem_full = bars + 2 * STAGES;                    // [ACC_BUFS] MMA -> epilogue
    uint64_t* tmem_empty = bars + 2 * STAGES + ACC_BUFS;        // [ACC_BUFS] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 2 * ACC_BUFS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tiles_n = a.N / BN, tiles_m = a.M / BM, n_tiles = tiles_m * tiles_n, kblocks = a.K / BK;
    // Wave quantisation (WIDE only): 512 tiles on 148 CTAs are 3.46 rounds = 4 rounds of time.  When the last, partial round holds at
    // most grid/2 tiles, each of them is split into two 128 x 128 halves (MMA N = 128, one TMA of B instead of two), so the tail costs
    // half a round: virtual tile ids [0, sched_full) are whole tiles, [sched_full, n_virtual) are halves (two consecutive ids per tile).
    uint32_t sched_full = n_tiles, n_virtual = n_tiles;
    if (WIDE) {
        const uint32_t whole = (n_tiles / gridDim.x) * gridDim.x, rem = n_tiles - whole;
        if (rem && 2u * rem <= gridDim.x) { sched_full = whole; n_virtual = whole + 2u * rem; }
    }
    auto decode = [&](uint32_t v, uint32_t& tm, uint32_t& n_off, uint32_t& bn_t) {
        uint32_t w = v, h = 0, tn;
        bn_t = BN;
        if (v >= sched_full) { w = sched_full + ((v - sched_full) >> 1); h = (v - sched_full) & 1u; bn_t = BN / 2; }
        tile_coords(w, tiles_m, tiles_n, GROUP_M, tm, tn);
        n_off = tn * BN + h * (BN / 2);
    };

    if (threadIdx.x == 0) {
        tma_prefetch_desc(map_a); tma_prefetch_desc(map_b);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < ACC_BUFS; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], EPI_THREADS); }
        fence_barrier_init();
    }
    if (warp == 2) {                                            // one warp allocates TMEM and later frees it
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ===== TMA producer =====
        uint32_t it = 0;
        const uint64_t pol_a = l2_policy_evict_last(), pol_b = l2_policy_evict_first();
        for (uint32_t tile = blockIdx.x; tile < n_virtual; tile += gridDim.x) {
            uint32_t tm, n_off, bn_t;
            decode(tile, tm, n_off, bn_t);
            const int m0 = (int)tm * BM, n0 = (int)n_off;
            const int b_loads = (int)bn_t / 128;                // the B box is {32 n, 32 k, 4 chunks} = 128 columns: two loads per wide tile
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                mbar_wait(&empty[s], ph ^ 1u);
                mbar_arrive_expect_tx(&full[s], A_STAGE + bn_t * BK * 4u);
                tma_load_2d_hint(sA + s * A_STAGE, map_a, &full[s], (int)(kb * BK), m0, pol_a);         // box {32 k, 128 m}
                for (int c = 0; c < b_loads; ++c)
                    tma_load_3d_hint(sB + s * B_STAGE + c * (4 * BK * 128), map_b, &full[s], 0, (int)(kb * BK), n0 / 32 + 4 * c, pol_b);
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp walks the pipeline converged, ONE elected lane issues; every MMA is issued NC times
        // into NC accumulators.  (A lone diverged thread makes ptxas wrap each UTC*MMA in an elect/branch loop and rebuild both
        // descriptors per instruction; hoisting the descriptor arithmetic leaves one UTCHMMA + one 64-bit add per MMA.)
        const bool leader = elect_one();
        uint32_t it = 0, tcount = 0;
        for (uint32_t tile = blockIdx.x; tile < n_virtual; tile += gridDim.x, ++tcount) {
            const uint32_t buf = tcount % ACC_BUFS, use = tcount / ACC_BUFS;
            const uint32_t bn_t = tile >= sched_full ? BN / 2 : BN;
            const uint32_t idesc = (G::IDESC & ~(0x3Fu << 17)) | ((bn_t >> 3) << 17);      // MMA N of this tile
            mbar_wait(&tmem_empty[buf], (use & 1u) ^ 1u);       // epilogue drained this accumulator set
            tc_fence_after();
            const uint32_t acc0 = tmem_base + buf * (uint32_t)(NC * BN);
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                if (leader) {
                    // A: K-major SW128, rows 128 B apart, 8-row groups 1024 B apart; advance 32 B per UMMA_K inside the swizzle row
                    const uint64_t da0 = smem_desc(smem_u32(sA + s * A_STAGE), 16, 1024, SWZ_128B);
                    // B: MN-major, 32B-atom swizzle: atom = 4 k-rows x 128 B (512 B, SBO); N chunks BK*128 B apart (LBO);
                    // one UMMA_K = 8 k-rows = 1024 B further down the chunk
                    const uint64_t db0 = smem_desc(smem_u32(sB + s * B_STAGE), BK * 128, 512, SWZ_128B_BASE32B);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t da = da0 + (uint64_t)((k * UMMA_K * 4) >> 4), db = db0 + (uint64_t)((k * 1024) >> 4);
                        const uint32_t acc = (kb | (uint32_t)k) ? 1u : 0u;
                        if (NC == 1) {
                            tc_mma_tf32(acc0, da, db, idesc, acc);
                        } else {                                // A stays in the collector across the replicas of this k-step
                            tc_mma_tf32_col<1>(acc0, da, db, idesc, acc);
                            if (NC == 3) tc_mma_tf32_col<2>(acc0 + BN, da, db, idesc, acc);
                            tc_mma_tf32_col<3>(acc0 + (NC - 1) * BN, da, db, idesc, acc);
                        }
                    }
                    tc_commit(&empty[s]);                       // smem slot free once these MMAs retire
                }
                __syncwarp();
            }
            if (leader) tc_commit(&tmem_full[buf]);             // accumulators complete
            __syncwarp();
        }
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> registers, vote, count, ONE store =====
        const int q = warp & 3;                                 // TMEM lane quarter this warp may touch
        const int half = (warp - 4) >> 2;                       // two warps per quarter, each takes half of the tile's columns
        const uint64_t pol_c = l2_policy_evict_first();
        Tally tally(a);
        uint32_t tcount = 0;
        for (uint32_t tile = blockIdx.x; tile < n_virtual; tile += gridDim.x, ++tcount) {
            uint32_t tm, n0, bn_t;
            decode(tile, tm, n0, bn_t);
            const uint32_t m0 = tm * BM;
            const uint32_t buf = tcount % ACC_BUFS, use = tcount / ACC_BUFS;
            mbar_wait(&tmem_full[buf], use & 1u);
            tc_fence_after();
            const uint32_t row = m0 + q * 32 + lane;
            const uint32_t lane_addr = tmem_base + buf * (uint32_t)(NC * BN) + ((uint32_t)(q * 32) << 16);
            epilogue_cols<NC, INJECT>(a, tally, lane_addr, (uint32_t)BN, row, n0, half * (int)(bn_t / 2), (half + 1) * (int)(bn_t / 2), pol_c);
            tc_fence_before();
            mbar_arrive(&tmem_empty[buf]);                      // EPI_THREADS arrivals release this accumulator set
        }
        tally.flush(a.counters);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
    }
}

}  // namespace gemm
}  // namespace xmr

#define XMR_GEMM_KERNEL(NC, INJ)                                                                         \
    extern "C" __global__ void __launch_bounds__(xmr::gemm::CTA_THREADS, 1)                                                 \
    xmr_gemm_tf32_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap map_a, \
                                    const __grid_constant__ CUtensorMap map_b) {                         \
        xmr::gemm::gemm_body<NC, INJ != 0>(a, &map_a, &map_b);                                           \
    }
XMR_GEMM_KERNEL(1, 0) XMR_GEMM_KERNEL(2, 0) XMR_GEMM_KERNEL(3, 0)
XMR_GEMM_KERNEL(1, 1) XMR_GEMM_KERNEL(2, 1) XMR_GEMM_KERNEL(3, 1)
// unprotected, N a multiple of 128 but not of 256: 128 x 128 tiles (shared-memory operands, two accumulator buffers)
#define XMR_GEMM_KERNEL_NARROW(INJ)                                                                      \
    extern "C" __global__ void __launch_bounds__(xmr::gemm::CTA_THREADS, 1)                                                 \
    xmr_gemm_tf32n_nc1_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap map_a, \
                                const __grid_constant__ CUtensorMap map_b) {                             \
        xmr::gemm::gemm_body<1, INJ != 0, false>(a, &map_a, &map_b);                                     \
    }
XMR_GEMM_KERNEL_NARROW(0) XMR_GEMM_KERNEL_NARROW(1)
