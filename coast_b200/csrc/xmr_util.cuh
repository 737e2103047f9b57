// xmr_util.cuh -- small service kernels of the runtime (counter reset, synthetic input).
#pragma once
#include "xmr_common.cuh"

// dst[i] = Philox4x32-10(ctr = {(word_base + i) / 4, 0, 0, 0}, key = {seed, 0})[(word_base + i) % 4]
// (SURVEY.md 8d: one counter-based generator so CPU oracle and GPU see identical bytes)
extern "C" __global__ void __launch_bounds__(256)
xmr_fill_philox(uint32_t* __restrict__ dst, unsigned long long n_words, unsigned long long word_base, uint32_t seed) {
    const unsigned long long first_blk = word_base >> 2;
    const unsigned long long last_blk = (word_base + n_words + 3ull) >> 2;   // exclusive
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long blk = first_blk + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; blk < last_blk; blk += stride) {
        xmr::u4 x = xmr::philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), 0u, 0u, seed, 0u);
        const uint32_t v[4] = {x.x, x.y, x.z, x.w};
        const unsigned long long w0 = blk << 2;
        if (w0 >= word_base && w0 + 4ull <= word_base + n_words && ((reinterpret_cast<uintptr_t>(dst + (w0 - word_base)) & 15u) == 0)) {
            *reinterpret_cast<uint4*>(dst + (w0 - word_base)) = make_uint4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                unsigned long long w = w0 + q;
                if (w >= word_base && w < word_base + n_words) dst[w - word_base] = v[q];
            }
        }
    }
}

extern "C" __global__ void xmr_counters_reset(unsigned long long* ctr) {
    if (threadIdx.x < XMR_CTR_COUNT) ctr[threadIdx.x] = threadIdx.x == XMR_CTR_FIRST ? ~0ull : 0ull;
}

// One record per SM that gets a CTA: {clock64(), %globaltimer [ns]} at out[2 * smid ..].  Two probes around a region give the
// AVERAGE SM clock the region really ran at (delta cycles / delta ns per SM) -- NVML's clocks.sm keeps reporting the nominal clock
// while the tensor kernels run ~15 % below it under the power limit (profiles/r02_gemm_*: ncu smsp__cycles_elapsed.avg.per_second).
extern "C" __global__ void xmr_clock_probe(unsigned long long* out) {
    if (threadIdx.x == 0) {
        unsigned smid;
        unsigned long long t;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        const unsigned long long c = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        out[2 * smid] = c;
        out[2 * smid + 1] = t;
    }
}
