// xmr_mm_tc.cuh -- protected EXACT integer matmul on the tensor cores (tcgen05.mma kind::i8).
//
// matrix_multiply() of the reference (tests/mm_common/mm_common_tmr.c:3-20, tests/matrixMultiply/matrixMultiply.c:95-112)
// is integer arithmetic modulo 2^32.  Split every u32 into four u8 limbs, a = sum_i a_i 2^(8i), b = sum_j b_j 2^(8j):
//     a*b mod 2^32 = sum_{i+j<=3} (a_i * b_j) << 8(i+j)
// so C = S0 + (S1 << 8) + (S2 << 16) + (S3 << 24) mod 2^32 with S_d = sum_{i+j=d} A_i . B_j  -- ten u8 x u8 GEMMs whose
// s32 accumulators are allowed to WRAP (tools/probe/tc_probe_i8.cu checks the tensor core wraps rather than saturates),
// which keeps every S_d exact modulo 2^32 for any K.  Bit-exact with the reference's own loops, at tensor-core rate.
//
// Data path:  xmr_mm_split_a / xmr_mm_split_bt (pre-pass, library scratch): A -> 4 u8 planes [l][M][K], B -> 4 TRANSPOSED
// u8 planes [l][N][K] (both K-major: the plain SWIZZLE_128B K-major descriptor, no MN-major special case);
// TMA (one 3-D box per operand per stage: {128 k, rows, 4 planes}) -> 2-stage ring; the elected lane of the MMA warp issues,
// per 32-byte k-step, the 10 limb-pair MMAs NC times into NC x 4 TMEM accumulators (S0..S3 per replica, BN columns each)
// (staging A in TMEM with tcgen05.cp + TS-mode MMAs works -- tools/probe/tc_probe_i8.cu -- but measured slower here);
// the epilogue recombines each replica's C from its four accumulators, votes element-wise (one mm_t vote per unit),
// counts, and stores ONE C tile.  Fault site s (`sum` after k-step s) is applied lazily and exactly as in xmr_mm_tiled.cuh.
#pragma once
#include "xmr_common.cuh"
#include "xmr_gemm_tf32.cuh"   // tcgen05 / TMA helpers (xmr::gemm::*)

namespace xmr {
namespace mmtc {

using namespace xmr::gemm;

constexpr int TBM = 128, TBK = 128;                 // 128 u8 of K = one 128-byte swizzle row = 4 MMAs of K=32
// ATMEM: stage each k-block's A limb planes into TMEM with tcgen05.cp and run the MMAs in TS mode (A from TMEM): every A slice
// is then fetched from shared memory once instead of by each of the up to 4 x NC MMAs that use it.
template <int NC, bool ATMEM> struct Geom {
    static constexpr int BN = ATMEM ? (NC == 1 ? 64 : 32) : (NC == 3 ? 32 : 64);   // accumulators (+128 columns of staged A) <= 512
    static constexpr uint32_t A_STAGE_B = 4u * TBM * TBK;            // 64 KiB: [plane][row][128 B]
    static constexpr uint32_t B_STAGE_B = 4u * BN * TBK;             // 16 / 32 KiB
    static constexpr int STAGES_ = 2;
    static constexpr uint32_t SMEM = STAGES_ * (A_STAGE_B + B_STAGE_B) + 1024 + 256;
    static constexpr uint32_t ACC_COLS = NC * 4 * BN;                // S0..S3 per replica
    static constexpr uint32_t A_COLS = ATMEM ? 4 * (TBK / 32) * 8 : 0;   // 4 planes x 4 k-steps x (32 bytes = 8 columns)
    static constexpr uint32_t TMEM = ACC_COLS + A_COLS <= 256 ? 256 : 512;
    static_assert(ACC_COLS + A_COLS <= 512, "TMEM budget");
};
// idesc: c_format S32 (2) [4,6); a/b format 0 = UNSIGNED 8 bit [7,10)/[10,13); both K-major; N>>3 [17,23); M>>4 [24,29)
template <int BN> struct IdescU8 { static constexpr uint32_t value = (2u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TBM >> 4) << 24); };

__device__ __forceinline__ void tc_mma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// A-operand collector usage as xmr::gemm::tc_mma_tf32_col: 1 = fill, 2 = use, 3 = lastuse (0 = plain)
template <int USAGE>
__device__ __forceinline__ void tc_mma_i8_col(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if (USAGE == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 2)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::use [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else if (USAGE == 3)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
    else
        tc_mma_i8(d_tmem, a_desc, b_desc, idesc, accumulate);
}
// A operand from TMEM (128 lanes x 8 columns = 128 rows x 32 bytes of K), B from shared memory
__device__ __forceinline__ void tc_mma_i8_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// shared memory (matrix descriptor, 128 rows x 256 bits) -> TMEM (128 lanes x 8 columns); SASS UTCCP
__device__ __forceinline__ void tc_cp_128x256b(uint32_t taddr, uint64_t s_desc) {
    asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(s_desc) : "memory");
}
__device__ __forceinline__ void tc_ld_32x8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
}

template <int NC, bool INJECT, bool ATMEM>
__device__ __forceinline__ void body(const xmr_args& a, const CUtensorMap* map_a, const CUtensorMap* map_b) {
    using G = Geom<NC, ATMEM>;
    constexpr int BN = G::BN, STAGES_ = G::STAGES_;
    extern __shared__ uint8_t smem_dyn[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023u) & ~(uintptr_t)1023u);
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES_ * G::A_STAGE_B;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES_ * (G::A_STAGE_B + G::B_STAGE_B));
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES_;
    uint64_t* tmem_full = bars + 2 * STAGES_;
    uint64_t* tmem_empty = bars + 2 * STAGES_ + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES_ + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tiles_n = a.N / BN, tiles_m = a.M / TBM, n_tiles = tiles_m * tiles_n, kblocks = a.K / TBK;
    // tile order: GROUP_M tile-rows per group, column-major inside (same L2 argument as the TF32 kernel)
    auto coords = [&](uint32_t tile, uint32_t& tm, uint32_t& tn) {
        const uint32_t per_group = GROUP_M * tiles_n, g = tile / per_group, w = tile - g * per_group;
        const uint32_t rows = min(GROUP_M, tiles_m - g * GROUP_M);
        tm = g * GROUP_M + w % rows; tn = w / rows;
    };

    if (threadIdx.x == 0) {
        tma_prefetch_desc(map_a); tma_prefetch_desc(map_b);
        for (int s = 0; s < STAGES_; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 128);
        fence_barrier_init();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(G::TMEM) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_a = tmem_base + G::ACC_COLS;            // ATMEM: staged A operand

    if (warp == 0 && lane == 0) {
        uint32_t it = 0;
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            uint32_t tm, tn; coords(tile, tm, tn);
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES_, ph = (it / STAGES_) & 1u;
                mbar_wait(&empty[s], ph ^ 1u);
                mbar_arrive_expect_tx(&full[s], G::A_STAGE_B + G::B_STAGE_B);
                tma_load_3d(sA + s * G::A_STAGE_B, map_a, &full[s], (int)(kb * TBK), (int)(tm * TBM), 0);   // box {128 k, 128 m, 4 planes}
                tma_load_3d(sB + s * G::B_STAGE_B, map_b, &full[s], (int)(kb * TBK), (int)(tn * BN), 0);    // box {128 k, BN n, 4 planes}
            }
        }
    } else if (warp == 1) {
        // The WHOLE warp walks the pipeline (converged), one elected lane issues.  With a lone diverged thread ptxas wraps
        // every UTCIMMA in an elect/branch loop and rebuilds both descriptors per MMA (~50 issue cycles each, measured:
        // 2.9 ms for the 4096^3 TMR problem, 3x the tensor time); hoisting the descriptor arithmetic and electing inside
        // converged code leaves one UTCIMMA + one add per MMA.
        constexpr uint32_t IDESC_U8 = IdescU8<BN>::value;
        const bool leader = elect_one();
        uint32_t it = 0, tcount = 0;
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
            mbar_wait(tmem_empty, (tcount & 1u) ^ 1u);
            tc_fence_after();
            for (uint32_t kb = 0; kb < kblocks; ++kb, ++it) {
                const uint32_t s = it % STAGES_, ph = (it / STAGES_) & 1u;
                mbar_wait(&full[s], ph);
                tc_fence_after();
                if (leader) {
                    // descriptors differ only in the 14-bit start-address field: base + (plane offset + k*32) >> 4
                    const uint64_t da0 = smem_desc(smem_u32(sA + s * G::A_STAGE_B), 16, 1024, SWZ_128B);
                    const uint64_t db0 = smem_desc(smem_u32(sB + s * G::B_STAGE_B), 16, 1024, SWZ_128B);
                    if (ATMEM) {   // tcgen05.cp and tcgen05.mma execute in issue order: this copy cannot overtake MMAs still reading block kb-1
#pragma unroll
                        for (int i = 0; i < 4; ++i)
#pragma unroll
                            for (int k = 0; k < TBK / 32; ++k)
                                tc_cp_128x256b(tmem_a + (i * (TBK / 32) + k) * 8, da0 + (uint64_t)((i * (TBM * TBK) + k * 32) >> 4));
                    }
                    if (!ATMEM) {
                        // Limb-major order: the (4 - i) x NC MMAs that multiply A limb i follow each other and keep that A slice in the
                        // tensor core's collector (fill ... use ... lastuse): 4 KiB of A per k-step and limb instead of per MMA.  The u8 MMA
                        // of N = BN reads 4 KiB of A + BN x 32 B of B per 16 tensor cycles -- 5x the shared-memory bandwidth without this.
                        // Integer accumulation is exact modulo 2^32, so the order of the limb products inside S_d does not matter; the
                        // first product into S_d of a tile is still (i = 0, j = d).
#pragma unroll
                        for (int k = 0; k < TBK / 32; ++k) {
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const uint64_t da = da0 + (uint64_t)((i * (TBM * TBK) + k * 32) >> 4);
                                const uint32_t acc = (kb | (uint32_t)k | (uint32_t)i) ? 1u : 0u;
#pragma unroll
                                for (int j = 0; j < 4 - i; ++j) {
                                    const uint64_t db = db0 + (uint64_t)((j * (BN * TBK) + k * 32) >> 4);
#pragma unroll
                                    for (int r = 0; r < NC; ++r) {
                                        const uint32_t dst = tmem_base + (r * 4 + (i + j)) * BN;
                                        const bool first = j == 0 && r == 0, last = j == 3 - i && r == NC - 1;
                                        if (first && last) tc_mma_i8(dst, da, db, IDESC_U8, acc);
                                        else if (first) tc_mma_i8_col<1>(dst, da, db, IDESC_U8, acc);
                                        else if (last) tc_mma_i8_col<3>(dst, da, db, IDESC_U8, acc);
                                        else tc_mma_i8_col<2>(dst, da, db, IDESC_U8, acc);
                                    }
                                }
                            }
                        }
                    } else
#pragma unroll
                    for (int k = 0; k < TBK / 32; ++k) {
#pragma unroll
                        for (int d = 0; d < 4; ++d) {            // diagonal d = i + j: shift 8d, accumulator S_d
#pragma unroll
                            for (int i = 0; i <= d; ++i) {
                                const int j = d - i;
                                const uint64_t db = db0 + (uint64_t)((j * (BN * TBK) + k * 32) >> 4);
                                const uint32_t acc = (kb | (uint32_t)k | (uint32_t)i) ? 1u : 0u;   // first MMA into S_d overwrites
#pragma unroll
                                for (int r = 0; r < NC; ++r)
                                    tc_mma_i8_ts(tmem_base + (r * 4 + d) * BN, tmem_a + (i * (TBK / 32) + k) * 8, db, IDESC_U8, acc);
                            }
                        }
                    }
                    tc_commit(&empty[s]);
                }
                __syncwarp();
            }
            if (leader) tc_commit(tmem_full);
            __syncwarp();
        }
    } else if (warp >= 4) {
        const int q = warp & 3;
        const uint32_t flags = a.flags;
        const bool majority = flags & COAST_F_MAJORITY_D;
        uint32_t* C = static_cast<uint32_t*>(a.out);
        const uint32_t* __restrict__ A32 = static_cast<const uint32_t*>(a.in);
        const uint32_t* __restrict__ B32 = static_cast<const uint32_t*>(a.aux);
        Tally tally(a);
        uint32_t tcount = 0;
        for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tcount) {
            uint32_t tm, tn; coords(tile, tm, tn);
            const uint32_t m0 = tm * TBM, n0 = tn * BN;
            mbar_wait(tmem_full, tcount & 1u);
            tc_fence_after();
            const uint32_t row = m0 + q * 32 + lane;
            const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 8) {
                uint32_t cr[3][8];
#pragma unroll
                for (int r = 0; r < NC; ++r) {
                    uint32_t s0[8], s1[8], s2[8], s3[8];
                    tc_ld_32x8(lane_addr + (r * 4 + 0) * BN + c0, s0);
                    tc_ld_32x8(lane_addr + (r * 4 + 1) * BN + c0, s1);
                    tc_ld_32x8(lane_addr + (r * 4 + 2) * BN + c0, s2);
                    tc_ld_32x8(lane_addr + (r * 4 + 3) * BN + c0, s3);
                    tc_wait_ld();
#pragma unroll
                    for (int e = 0; e < 8; ++e) cr[r][e] = s0[e] + (s1[e] << 8) + (s2[e] << 16) + (s3[e] << 24);   // mod 2^32
                }
                uint32_t o[8];
                const unsigned long long local0 = (unsigned long long)row * a.N + n0 + c0;
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    uint32_t r0 = cr[0][e], r1 = NC > 1 ? cr[1][e] : r0, r2 = NC > 2 ? cr[2][e] : r0;
                    if (INJECT) {
                        Fault f = fault_for_unit(a, NC, local0 + e, [](uint32_t) { return 32u; });
                        if (f.active) {
                            tally.injected++;
                            uint32_t part = 0;                  // S_s = partial sum over k <= site, from the original u32 operands
                            for (uint32_t k = 0; k <= f.site; ++k) part += __ldg(A32 + (size_t)row * a.K + k) * __ldg(B32 + (size_t)k * a.N + n0 + c0 + e);
                            const uint32_t mk = 1u << f.bit, delta = (part & mk) ? (0u - mk) : mk;
                            if (f.replica == 0) r0 += delta; else if (f.replica == 1) r1 += delta; else r2 += delta;
                        }
                    }
                    uint32_t vote = r0, bad = 0;
                    if (NC == 2) bad = r0 != r1;
                    if (NC == 3) {
                        const bool c01 = r0 == r1, c02 = r0 == r2;
                        vote = majority ? ((r0 & r1) | (r0 & r2) | (r1 & r2)) : (c01 ? r0 : r2);
                        bad = (c01 && c02) ? 0u : 1u;
                    }
                    o[e] = vote;
                    tally.unit_exit<NC>(bad, 1u, flags, a.unit_base + local0 + e);
                }
                uint32_t* dst = C + (size_t)row * a.N + n0 + c0;
                *reinterpret_cast<uint4*>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
                *reinterpret_cast<uint4*>(dst + 4) = make_uint4(o[4], o[5], o[6], o[7]);
            }
            tc_fence_before();
            mbar_arrive(tmem_empty);
        }
        tally.flush(a.counters);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(G::TMEM) : "memory");
    }
}

}  // namespace mmtc
}  // namespace xmr

// ---- limb-split pre-pass ---------------------------------------------------------------------------------------
// A (u32, rows x K, row-major) -> planes[l][row][k] (u8).  One thread = 4 consecutive k of one row.
extern "C" __global__ void __launch_bounds__(256)
xmr_mm_split_a(const uint32_t* __restrict__ A, uint8_t* __restrict__ planes, unsigned long long rows, unsigned long long K) {
    const unsigned long long quads = rows * K / 4ull, stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += stride) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(A) + q);
        const uint32_t lo = __byte_perm(v.x, v.y, 0x5140u);        // x.b0 y.b0 x.b1 y.b1  (interleave low halves)
        const uint32_t hi = __byte_perm(v.x, v.y, 0x7362u);        // x.b2 y.b2 x.b3 y.b3
        const uint32_t lo2 = __byte_perm(v.z, v.w, 0x5140u), hi2 = __byte_perm(v.z, v.w, 0x7362u);
        uint32_t* p = reinterpret_cast<uint32_t*>(planes);
        const unsigned long long plane = rows * K / 4ull;
        p[q] = __byte_perm(lo, lo2, 0x5410u);                      // plane 0: b0 of x,y,z,w
        p[plane + q] = __byte_perm(lo, lo2, 0x7632u);              // plane 1
        p[2ull * plane + q] = __byte_perm(hi, hi2, 0x5410u);       // plane 2
        p[3ull * plane + q] = __byte_perm(hi, hi2, 0x7632u);       // plane 3
    }
}
// B (u32, K x N, row-major) -> planes[l][n][k] (u8, TRANSPOSED so the MMA's B operand is K-major).  32 x 32 tiles via smem.
extern "C" __global__ void __launch_bounds__(256)
xmr_mm_split_bt(const uint32_t* __restrict__ B, uint8_t* __restrict__ planes, unsigned int K, unsigned int N) {
    __shared__ uint32_t tile[32][33];
    const unsigned int tiles_n = N / 32u, tiles_k = K / 32u;
    for (unsigned int t = blockIdx.x; t < tiles_n * tiles_k; t += gridDim.x) {
        const unsigned int k0 = (t / tiles_n) * 32u, n0 = (t % tiles_n) * 32u;
        for (int i = threadIdx.x; i < 1024; i += 256) tile[i >> 5][i & 31] = __ldg(B + (size_t)(k0 + (i >> 5)) * N + n0 + (i & 31));
        __syncthreads();
        const int n = threadIdx.x >> 3, kq = threadIdx.x & 7;      // 32 n x 8 k-quads
        const uint32_t w0 = tile[kq * 4][n], w1 = tile[kq * 4 + 1][n], w2 = tile[kq * 4 + 2][n], w3 = tile[kq * 4 + 3][n];
        const uint32_t lo = __byte_perm(w0, w1, 0x5140u), hi = __byte_perm(w0, w1, 0x7362u);
        const uint32_t lo2 = __byte_perm(w2, w3, 0x5140u), hi2 = __byte_perm(w2, w3, 0x7362u);
        const size_t plane = (size_t)N * K, off = (size_t)(n0 + n) * K + k0 + kq * 4;
        *reinterpret_cast<uint32_t*>(planes + off) = __byte_perm(lo, lo2, 0x5410u);
        *reinterpret_cast<uint32_t*>(planes + plane + off) = __byte_perm(lo, lo2, 0x7632u);
        *reinterpret_cast<uint32_t*>(planes + 2 * plane + off) = __byte_perm(hi, hi2, 0x5410u);
        *reinterpret_cast<uint32_t*>(planes + 3 * plane + off) = __byte_perm(hi, hi2, 0x7632u);
        __syncthreads();
    }
}

#define XMR_MMTC_KERNEL(NC, INJ)                                                                         \
    extern "C" __global__ void __launch_bounds__(256, 1)                                                 \
    xmr_mm_u32_tc_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap map_a, \
                                    const __grid_constant__ CUtensorMap map_b) {                         \
        xmr::mmtc::body<NC, INJ != 0, false>(a, &map_a, &map_b);                                         \
    }                                                                                                    \
    extern "C" __global__ void __launch_bounds__(256, 1)                                                 \
    xmr_mm_u32_tct_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap map_a, \
                                     const __grid_constant__ CUtensorMap map_b) {                        \
        xmr::mmtc::body<NC, INJ != 0, true>(a, &map_a, &map_b);                                          \
    }
XMR_MMTC_KERNEL(1, 0) XMR_MMTC_KERNEL(2, 0) XMR_MMTC_KERNEL(3, 0)
XMR_MMTC_KERNEL(1, 1) XMR_MMTC_KERNEL(2, 1) XMR_MMTC_KERNEL(3, 1)
