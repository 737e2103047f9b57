// xmr_mm_tiled.cuh -- protected exact integer matmul, register-tiled (the fast path of xmr_mm.cuh).
//
// Same arithmetic as matrix_multiply() (tests/mm_common/mm_common_tmr.c:3-20): r[i][j] = sum_k f[i][k]*s[k][j]
// with the `unsigned long sum` truncated to 32 bits at the store, i.e. exact modulo 2^32 (IMAD).
// Segmented replica layout (-s): the CTA has NC x 128 threads; thread t of replica r = t/128 is "virtual thread"
// vt = t%128 and ALL replicas of a vt compute the same 8x8 micro-tile of a 64 x 128 C tile from the SAME shared-memory
// operand tiles (one staged copy, read NC times).  SoR exit: replicas 1,2 publish their 64 accumulators through shared
// memory, replica 0 votes every element (one mm_t vote per unit) and stores the tile once.
// Fault site s (= `sum` after k-step s) is applied exactly but lazily: a flip of bit b in the partial sum S_s changes the
// final sum by +2^b or -2^b (mod 2^32) depending on bit b of S_s, so only faulted elements recompute a partial dot product.
#pragma once
#include "xmr_common.cuh"

namespace xmr {
namespace mmt {

constexpr int BM = 64, BN = 128, BK = 16, VT = 128;

__device__ __forceinline__ Voted vote3(uint32_t x, uint32_t r1, uint32_t r2, int nc, bool majority) {
    Voted v{x, 0u};
    if (nc == 2) v.bad = x != r1;
    if (nc == 3) {
        const bool c01 = x == r1, c02 = x == r2;
        v.vote = majority ? ((x & r1) | (x & r2) | (r1 & r2)) : (c01 ? x : r2);
        v.bad = (c01 && c02) ? 0u : 1u;
    }
    return v;
}

template <int NC, bool INJECT>
__device__ __forceinline__ void body(const xmr_args& a) {
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* As = smem;                        // [2][BK][BM]   (k-major: transposed on the way in)
    uint32_t* Bs = smem + 2 * BK * BM;          // [2][BK][BN]
    uint32_t* ex = smem;                        // epilogue: [NC-1][64][VT], reuses the operand buffers (64 KiB)
    const int tid = threadIdx.x, r = tid / VT, vt = tid % VT;
    const int tx = vt & 15, ty = vt >> 4;        // micro-tile: rows {ty*4+i, 32+ty*4+i}, cols {tx*4+j, 64+tx*4+j}
    const uint32_t N = a.N, K = a.K;
    const uint32_t tiles_n = N / BN;
    const uint32_t m0 = (blockIdx.x / tiles_n) * BM, n0 = (blockIdx.x % tiles_n) * BN;
    const uint32_t* __restrict__ A = static_cast<const uint32_t*>(a.in);
    const uint32_t* __restrict__ B = static_cast<const uint32_t*>(a.aux);
    constexpr int NT = NC * VT;
    constexpr int A_V4 = BM * BK / 4, B_V4 = BK * BN / 4;          // 256 + 512 uint4 per k-tile
    constexpr int PER = (A_V4 + B_V4 + NT - 1) / NT;

    uint32_t acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0u;

    uint4 pre[PER];
    auto gload = [&](uint32_t k0) {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = tid + p * NT;
            if (q < A_V4) {                       // A: row q/4 of the tile, k-quad q%4
                pre[p] = __ldg(reinterpret_cast<const uint4*>(A + (size_t)(m0 + q / 4) * K + k0 + (q % 4) * 4));
            } else if (q < A_V4 + B_V4) {         // B: k-row (q-A)/32, column quad (q-A)%32
                const int b = q - A_V4;
                pre[p] = __ldg(reinterpret_cast<const uint4*>(B + (size_t)(k0 + b / 32) * N + n0 + (b % 32) * 4));
            }
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int q = tid + p * NT;
            if (q < A_V4) {
                uint32_t* d = As + buf * BK * BM + ((q % 4) * 4) * BM + q / 4;
                d[0] = pre[p].x; d[BM] = pre[p].y; d[2 * BM] = pre[p].z; d[3 * BM] = pre[p].w;
            } else if (q < A_V4 + B_V4) {
                const int b = q - A_V4;
                *reinterpret_cast<uint4*>(Bs + buf * BK * BN + (b / 32) * BN + (b % 32) * 4) = pre[p];
            }
        }
    };

    const uint32_t ktiles = K / BK;
    gload(0);
    sstore(0);
    __syncthreads();
    for (uint32_t kt = 0; kt < ktiles; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < ktiles) gload((kt + 1) * BK);
        const uint32_t* as = As + buf * BK * BM;
        const uint32_t* bs = Bs + buf * BK * BN;
#pragma unroll
        for (int k = 0; k < BK; ++k) {                          // :12-14
            const uint4 a0 = *reinterpret_cast<const uint4*>(as + k * BM + ty * 4);
            const uint4 a1 = *reinterpret_cast<const uint4*>(as + k * BM + 32 + ty * 4);
            const uint4 b0 = *reinterpret_cast<const uint4*>(bs + k * BN + tx * 4);
            const uint4 b1 = *reinterpret_cast<const uint4*>(bs + k * BN + 64 + tx * 4);
            const uint32_t av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const uint32_t bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] += av[i] * bv[j];
        }
        if (kt + 1 < ktiles) sstore(buf ^ 1);
        __syncthreads();
    }

    Tally tally(a);
    const bool majority = a.flags & COAST_F_MAJORITY_D;
    auto row_of = [&](int i) { return m0 + (i < 4 ? ty * 4 + i : 32 + ty * 4 + (i - 4)); };
    auto col_of = [&](int j) { return n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4)); };

    if (INJECT) {
#pragma unroll 1
        for (int e = 0; e < 64; ++e) {
            const int i = e >> 3, j = e & 7;
            const uint32_t row = row_of(i), col = col_of(j);
            const unsigned long long local = (unsigned long long)row * N + col;
            Fault f = fault_for_unit(a, NC, local, [](uint32_t) { return 32u; });
            if (!f.active) continue;
            if (r == 0) tally.injected++;
            if ((int)f.replica != r) continue;
            uint32_t part = 0;                                  // S_s = sum over k <= site
            for (uint32_t k = 0; k <= f.site; ++k) part += __ldg(A + (size_t)row * K + k) * __ldg(B + (size_t)k * N + col);
            const uint32_t mk = 1u << f.bit;
            const uint32_t delta = (part & mk) ? (0u - mk) : mk;  // (S ^ mk) - S
#pragma unroll
            for (int ii = 0; ii < 8; ++ii)
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) acc[ii][jj] += (ii == i && jj == j) ? delta : 0u;
        }
    }

    // SoR exit
    if (NC > 1) {
        __syncthreads();                                        // operand buffers are dead: reuse as exchange
        if (r > 0) {
#pragma unroll
            for (int e = 0; e < 64; ++e) ex[((r - 1) * 64 + e) * VT + vt] = acc[e >> 3][e & 7];
        }
        __syncthreads();
    }
    if (r == 0) {
        uint32_t* C = static_cast<uint32_t*>(a.out);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t row = row_of(i);
            uint32_t o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int e = i * 8 + j;
                const uint32_t r1 = NC > 1 ? ex[e * VT + vt] : 0u, r2 = NC > 2 ? ex[(64 + e) * VT + vt] : 0u;
                const Voted v = vote3(acc[i][j], r1, r2, NC, majority);
                o[j] = v.vote;
                tally.unit_exit<NC>(v.bad, 1u, a.flags, a.unit_base + (unsigned long long)row * N + col_of(j));
            }
            *reinterpret_cast<uint4*>(C + (size_t)row * N + n0 + tx * 4) = make_uint4(o[0], o[1], o[2], o[3]);        // :16
            *reinterpret_cast<uint4*>(C + (size_t)row * N + n0 + 64 + tx * 4) = make_uint4(o[4], o[5], o[6], o[7]);
        }
    }
    tally.flush(a.counters);
}

}  // namespace mmt
}  // namespace xmr

#define XMR_MMT_KERNEL(NC, INJ)                                                                          \
    extern "C" __global__ void __launch_bounds__(NC * 128)                                               \
    xmr_mm_u32_tiled_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a) { xmr::mmt::body<NC, INJ != 0>(a); }
XMR_MMT_KERNEL(1, 0) XMR_MMT_KERNEL(2, 0) XMR_MMT_KERNEL(3, 0)
XMR_MMT_KERNEL(1, 1) XMR_MMT_KERNEL(2, 1) XMR_MMT_KERNEL(3, 1)
