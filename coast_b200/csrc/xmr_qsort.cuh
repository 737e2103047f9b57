// xmr_qsort.cuh -- protected quick_sort() (tests/quicksort/quicksort.c:121-136 of byuccl/coast; SURVEY.md 8f-4).
//
// The one workload whose branches depend on DATA, so its sync points are the conditional-branch conditions inside the
// loops (populateSyncPoints synchronization.cpp:146-155, syncTerminator :741-1113, the same select voter :934-938):
// the NC replica lanes of a unit run in lockstep, every data-dependent condition (`A[i] < pivot`, `A[j] > pivot`) is voted
// with sub-warp shuffles over the unit's lane group and ALL replicas follow the voted branch; each replica swaps inside
// its own private copy of the array (memory replication).  The copies live in a library-owned, stream-ordered scratch
// buffer (a.aux): one NC x L slot per unit, element-major with the NC replicas of an element adjacent
// (Au[e * NC + r]).  The i++ / j-- scans of :126-127 then walk one 128-byte line per 32/NC elements, the replica lanes of
// a unit share that line, and the ~2 active lines per unit stay in L1; thread-local memory (32-way interleaved) put every
// element of a lane in a different line (r01: 17.8 ms for 65 536 x 580 ints under TMR, DRAM-latency bound), and a
// lane-major slot per replica tripled the lines a TMR warp touches (L1 thrash at 44 warps per SM: 16-21 ms).
// SoR exit: one vote per stored element.
// Unit = one array of L = unit_bytes/4 ints (L <= 1024; the reference sorts 580).  Recursion = explicit stack, left first.
// Fault sites: s < 32L: the value loaded for the s-th executed data comparison; 32L <= s < 33L: element s-32L of the
// replica's private copy before sorting.  The CPU checker under oracle/ uses the identical enumeration, guards and order.
#pragma once
#include "xmr_common.cuh"

namespace xmr {

constexpr int QS_MAX = 1024;

// Execution scheme: a per-unit STATE MACHINE stepped by one uniform warp loop.  Written as the nested loops of :121-136,
// the units of a warp wait for each other at every loop exit (scan lengths and partition sizes differ wildly between
// arrays), which left ~1 lane group in 10 busy (r01: 16 ms TMR, issue-bound on serialised paths).  Here every iteration
// of the ONE loop advances EVERY unit by one step of its own control flow:
//   SCAN_I  one `at(i) < pivot` test of :126      SCAN_J  one `at(j) > pivot` test of :127, then :128-131 when it fails
//   POP     `quick_sort(A + i, len - i)` of :135 taken off the explicit stack (the left call :134 is entered directly)
// The data-dependent conditions of all units are voted with ONE warp ballot per iteration (each lane group reads its own
// NC bits).  The order of compare events, votes and swaps of a unit is exactly that of the nested loops, so the event
// numbering of the fault sites and every counter are unchanged (same oracle, same tests).
enum : uint32_t { QS_POP = 0u, QS_SCAN_I = 1u, QS_SCAN_J = 2u, QS_DONE = 3u };

template <int NC, bool INJECT>
__device__ __forceinline__ void qsort_body(const xmr_args& a) {
    constexpr int UPW = Lanes<NC>::kUnitsPerWarp;
    const int lane = threadIdx.x & 31;
    const bool spare = NC == 3 && lane >= 30;                   // the two idle TMR lanes only take part in the ballots
    const int u = spare ? 0 : lane / NC, r = spare ? 0 : lane % NC, base = u * NC;
    const uint32_t gmask = spare ? 0u : (((1u << NC) - 1u) << base);
    const unsigned long long gwarp = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const unsigned long long n_wtiles = (a.n_units + UPW - 1) / UPW;
    const uint32_t L = a.unit_bytes >> 2;
    const bool majority = (a.flags & COAST_F_MAJORITY_D) != 0;
    Tally tally(a);
    int32_t* const Au = static_cast<int32_t*>(const_cast<void*>(a.aux)) + (gwarp * 32ull + (unsigned)base) * L;   // this unit's NC x L slot
    auto at = [&](uint32_t e) -> int32_t& { return Au[e * NC + (uint32_t)r]; };                  // element e of this replica
    uint32_t stack[QS_MAX];                                     // (off << 16) | len, len <= 1024 needs 11 bits
    for (unsigned long long wt = gwarp; wt < n_wtiles; wt += nwarps) {
        const unsigned long long local = wt * UPW + u;
        const bool valid = !spare && local < a.n_units;
        uint32_t fsite = 0xFFFFFFFFu, fmask = 0u;
        if (valid) {
            const int32_t* src = static_cast<const int32_t*>(a.in) + local * L;
            for (uint32_t e = 0; e < L; ++e) at(e) = __ldg(src + e);
            if (INJECT) {
                Fault f = fault_for_unit(a, NC, local, [](uint32_t) { return 32u; });
                if (f.active) {
                    if (r == 0) tally.injected++;
                    if ((int)f.replica == r) { fsite = f.site; fmask = 1u << f.bit; }
                }
                if (fsite >= 32u * L && fsite != 0xFFFFFFFFu) at(fsite - 32u * L) ^= (int32_t)fmask;
            }
        }
        uint32_t ndis = 0, syncs = 0, ev = 0;                   // disagreeing branch votes, executed sync points, compare events
        uint32_t phase = valid ? QS_POP : QS_DONE;
        uint32_t off = 0, len = 0;
        int32_t pivot = 0, i = 0, j = 0;
        int sp = 0;
        if (valid) stack[sp++] = L;                             // quick_sort(A, n): off = 0
        __syncwarp();
        while (__any_sync(0xFFFFFFFFu, phase != QS_DONE)) {
            // ---- the data-dependent condition of this step (false for units that are between partitions)
            const bool scan_i = phase == QS_SCAN_I, scan_j = phase == QS_SCAN_J;
            bool c = false;
            if (scan_i || scan_j) {
                int32_t v = at(off + (uint32_t)(scan_i ? i : j));
                if (INJECT && fsite == ev) v ^= (int32_t)fmask;
                ++ev;
                c = scan_i ? (v < pivot) : (v > pivot);
                if (scan_i ? (i >= (int32_t)len - 1) : (j <= 0)) c = false;   // trap guard: a mis-steered scan stops at the partition edge
            }
            const uint32_t bal = __ballot_sync(0xFFFFFFFFu, c);
            bool voted = c;
            if (NC >= 2) {
                const uint32_t c0 = (bal >> base) & 1u, c1 = (bal >> (base + 1)) & 1u;
                if (NC == 2) { if (c0 != c1) ndis++; voted = c0 != 0u; }
                else {
                    const uint32_t c2 = (bal >> (base + 2)) & 1u;
                    const bool c01 = c0 == c1, c02 = c0 == c2;
                    if (!(c01 && c02)) ndis++;
                    voted = (majority ? ((c0 & c1) | (c0 & c2) | (c1 & c2)) : (c01 ? c0 : c2)) != 0u;
                }
            }
            // ---- advance this unit by one step
            if (scan_i) {
                syncs++;
                if (voted) i++; else phase = QS_SCAN_J;         // while (at(i) < pivot) i++;   :126
            } else if (scan_j) {
                syncs++;
                if (voted) j--;                                 // while (at(j) > pivot) j--;   :127
                else {
                    syncs++;                                    // if (i >= j) break;   :128 -- indices always agree
                    if (i < j) {
                        const int32_t t = at(off + (uint32_t)i); at(off + (uint32_t)i) = at(off + (uint32_t)j); at(off + (uint32_t)j) = t;   // :129-131, own copy
                        i++; j--; phase = QS_SCAN_I;            // for (;; i++, j--)   :125
                    } else {
                        if (i < 1) i = 1;
                        if (i > (int32_t)len - 1) i = (int32_t)len - 1;
                        stack[sp++] = ((off + (uint32_t)i) << 16) | (len - (uint32_t)i);   // quick_sort(A + i, len - i)  :135 (later)
                        len = (uint32_t)i;                                                  // quick_sort(A, i)            :134 (now)
                        syncs++;                                // its `if (len < 2) return;`   :122
                        if (len < 2) phase = QS_POP;
                        else { pivot = at(off + len / 2); i = 0; j = (int32_t)len - 1; phase = QS_SCAN_I; }   // :123-125
                    }
                }
            } else if (phase == QS_POP) {
                if (sp == 0) phase = QS_DONE;
                else {
                    const uint32_t top = stack[--sp];
                    off = top >> 16; len = top & 0xFFFFu;
                    syncs++;                                    // `if (len < 2) return;`   :122
                    if (len >= 2) { pivot = at(off + len / 2); i = 0; j = (int32_t)len - 1; phase = QS_SCAN_I; }
                }
            }
        }
        if (valid) {
            // SoR exit: one vote per stored element
            int32_t* dst = static_cast<int32_t*>(a.out) + local * L;
            uint32_t bad = 0;
            for (uint32_t e = 0; e < L; ++e) {
                const int32_t x = at(e);
                int32_t v = x;
                if (NC >= 2) {
                    const int32_t r1 = __shfl_sync(gmask, x, base + 1);
                    const int32_t r0 = __shfl_sync(gmask, x, base);
                    if (NC == 2) { bad += r0 != r1; v = r0; }
                    else {
                        const int32_t r2 = __shfl_sync(gmask, x, base + 2);
                        const bool c01 = r0 == r1, c02 = r0 == r2;
                        v = majority ? ((r0 & r1) | (r0 & r2) | (r1 & r2)) : (c01 ? r0 : r2);
                        bad += (c01 && c02) ? 0u : 1u;
                    }
                }
                if (r == 0) dst[e] = v;
            }
            if (r == 0) {
                const unsigned long long gunit = a.unit_base + local;
                if (NC == 3) {
                    if (a.flags & COAST_F_COUNT_ERRORS_D) {
                        tally.errors += bad + ndis;
                        if (a.flags & COAST_F_COUNT_SYNCS_D) tally.syncs += syncs + L;
                    }
                } else if (NC == 2) {
                    tally.dwc += (bad || ndis) ? 1u : 0u;
                }
                const uint32_t dis = bad + ndis;
                if (NC > 1 && dis && gunit < tally.first) tally.first = gunit;
                if (tally.status) tally.status[local] = (unsigned char)(NC > 1 ? (dis > 255u ? 255u : dis) : 0u);
            }
        }
        __syncwarp();
    }
    tally.flush(a.counters);
}

}  // namespace xmr

#define XMR_QSORT_KERNEL(NC, INJ)                                                                        \
    extern "C" __global__ void __launch_bounds__(128)                                                    \
    xmr_qsort_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a) { xmr::qsort_body<NC, INJ != 0>(a); }
XMR_QSORT_KERNEL(1, 0) XMR_QSORT_KERNEL(2, 0) XMR_QSORT_KERNEL(3, 0)
XMR_QSORT_KERNEL(1, 1) XMR_QSORT_KERNEL(2, 1) XMR_QSORT_KERNEL(3, 1)
