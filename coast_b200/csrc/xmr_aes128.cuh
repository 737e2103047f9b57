// xmr_aes128.cuh -- protected AES-128 single-block (tests/aes/TI_aes_128.c:107-231 of byuccl/coast)
//
// Unit = one 16-byte block -> 16 bytes.  SoR exit = the 16 u8 state bytes (:224-229): 16 votes.
// ONE table-driven body, four instantiations per (NC, injector):
//   enc   : encrypt, one ECB key expanded once per lane (BASELINE config 3)
//   dec   : decrypt, one key (round keys and their InvMixColumns images expanded once per lane)
//   enck / deck : per-unit keys from d_aux with the on-the-fly key schedule of the reference
//           (forward :214-221, to-the-last-round-key :112-129, inverse :133-141), optional write-back of what
//           aes_enc_dec() leaves in key[] (the last round key after encrypt, the original key after decrypt)
// Column formulation of the same rounds.  Encrypt: AddRoundKey-then-SubBytes (:143-146), ShiftRows (:147-166),
// MixColumns (:169-184) = four TE rows XORed.  Decrypt: the reference's iteration is [InvMixColumns (:169-184 with the
// :172-177 pre-multiply)] -> InvShiftRows (:187-206) -> InvSubBytes ^ key (:208-211); InvMixColumns is linear, so the
// kernel carries v = InvMixColumns(state) between iterations: v' = TD rows(v) ^ InvMixColumns(round key), and the last
// iteration ends with plain InvSubBytes ^ rk0.
// All tables are replicated 32x in shared memory (row x holds one copy per lane) so every lookup is bank-conflict free
// whatever the data and its address is ONE byte-permute; blocks arrive through the TMA tile ring.
// Fault sites (identical in oracle/): 0..15 = state byte as loaded; 16+16r+i = state[i] at the bottom of main-loop
// iteration r (:132-223).  A flip there is XOR-linear through the following AddRoundKey (and, for decrypt, through the
// following InvMixColumns), which is why the kernel can apply it to its fused values.
// Injector (r02, profiles/r02_aes_injector.md): the Philox draw of a unit is evaluated by ONE of its replica lanes and shuffled to the
// others; a unit whose flip lands mid-round is not finished in the tile loop but queued per warp and done in one pass after the
// last tile (aes_drain_deferred), because the code that applies such a flip is cold exactly because it is rare; the tile ring has no
// CTA-wide barrier (AesRing), so warps do not advance in lock-step.  DWC, 2^24 blocks, p = 2^-10: 0.740 ms vs 0.6845 ms without.
#pragma once
#include "xmr_common.cuh"
#include "aes_tables.inc"

namespace xmr {

// ---- geometry ----------------------------------------------------------------------------------
// 512-thread CTAs, one per SM.  Shared-memory WINDOW layout (absolute shared::cta addresses):
//   [dyn base .. 0x10000)  TMA tile ring (2 stages)
//   [0x10000 .. 0x20000)   row x (256 B): T0[x] replicated over 32 lanes | T1[x] = rotl8  replicated over 32 lanes
//   [0x20000 .. 0x30000)   row x (256 B): T2[x] = rotl16 x 32 lanes     | T3[x] = rotl24 x 32 lanes
//   [0x30000 .. 0x38000)   decrypt only, row x (128 B): (InvS[x], S[x], InvS[x], S[x]) replicated over 32 lanes
// T = TE (encrypt) or TD (decrypt).  Row stride 256 B + 64 KiB alignment make the lookup address ONE byte-permute:
//   addr = PRMT(t, lanebase) = lanebase.b3 : lanebase.b2 : byte_k(t) : lanebase.b0,  lanebase = table | half | lane*4
// and bank = lane for every lane whatever the data -> no shared-memory bank conflicts, no rotates, no LEA.  The 128-byte
// rows of the third window cost one extra shift: addr = PRMT(t, 2*lanebase) >> 1.
constexpr int AES_THREADS = 512, AES_WARPS = 16;
constexpr uint32_t AES_TAB01 = 0x10000u, AES_TAB23 = 0x20000u, AES_SIS = 0x30000u;
constexpr uint32_t AES_WINDOW_END_ENC = 0x30000u, AES_WINDOW_END_DEC = 0x38000u;
template <int NC> struct AesGeom { static constexpr int J = NC == 1 ? 2 : 4; static constexpr int TROWS = AES_WARPS * Lanes<NC>::kUnitsPerWarp * J; };

// Input ring of the AES kernels: 3 stages, full[] (TMA -> warps) and empty[] (warps -> the issuing thread) mbarriers and NO
// CTA-wide barrier in the tile loop.  r02 ablation (profiles/r02_aes_injector_ablation.txt): with the r01 ring's __syncthreads()
// per tile the 16 warps of a CTA advance in lock-step, so (a) the ALU-only Philox phase of the injector ran while the
// shared-memory pipe idled (+14.5 % with a plan that never hits) and (b) ONE warp on the rare hook path stalled the other 15
// for ~2 400 cycles at the next barrier (+0.13 ms at p = 2^-10).  Here a warp releases a stage as soon as its rows are in
// registers and runs up to two tiles ahead of the slowest warp; thread 0 refills a stage once all 16 warps have released it.
constexpr int AES_STAGES = 3;
template <int TILE_ROWS>
struct AesRing {
    static constexpr int pick_loads() { int l = (TILE_ROWS + 255) / 256; while (TILE_ROWS % l) ++l; return l; }
    static constexpr int LOADS = pick_loads();
    static constexpr int BOX_ROWS = TILE_ROWS / LOADS;
    static constexpr uint32_t TILE_BYTES = (uint32_t)TILE_ROWS * 16u;
    static constexpr uint32_t STAGE_STRIDE = (TILE_BYTES + 1023u) & ~1023u;
    static constexpr uint32_t SMEM_BYTES = AES_STAGES * STAGE_STRIDE + 128;
    uint8_t* tiles; uint64_t* full; uint64_t* empty; const CUtensorMap* tmap; uint32_t pack_shift;
    __device__ __forceinline__ void init(uint8_t* smem, const CUtensorMap* map, uint32_t row_pack_shift) {
        tiles = smem; tmap = map; pack_shift = row_pack_shift;
        full = reinterpret_cast<uint64_t*>(smem + AES_STAGES * STAGE_STRIDE);
        empty = full + AES_STAGES;
        if (threadIdx.x == 0) {
            tma_prefetch_desc(map);
#pragma unroll
            for (int s = 0; s < AES_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], AES_WARPS); }
            fence_barrier_init();
        }
        __syncthreads();
    }
    __device__ __forceinline__ void issue(uint32_t it, uint32_t tile) {           // thread 0 only
        const uint32_t stage = it % AES_STAGES;
        mbar_arrive_expect_tx(&full[stage], TILE_BYTES);
#pragma unroll
        for (int l = 0; l < LOADS; ++l)
            tma_load_2d(tiles + stage * STAGE_STRIDE + l * BOX_ROWS * 16, tmap, &full[stage], 0, (int)((tile * TILE_ROWS + l * BOX_ROWS) >> pack_shift));
    }
    __device__ __forceinline__ const uint8_t* wait_full(uint32_t it) {
        mbar_wait(&full[it % AES_STAGES], (it / AES_STAGES) & 1u);
        return tiles + (it % AES_STAGES) * STAGE_STRIDE;
    }
    __device__ __forceinline__ void release(uint32_t it, int lane) {              // whole warp: its rows of tile `it` are in registers
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&empty[it % AES_STAGES])) : "memory");
    }
    __device__ __forceinline__ void wait_empty(uint32_t it) {                     // every warp has released the stage tile `it` used
        mbar_wait(&empty[it % AES_STAGES], (it / AES_STAGES) & 1u);
    }
};

__device__ __forceinline__ uint32_t lds32(uint32_t saddr) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr)); return v; }
// table row of byte k of t: splice that byte into byte 1 of the lane's base address
template <int K> __device__ __forceinline__ uint32_t tab(uint32_t lb, uint32_t t) { return lds32(__byte_perm(t, lb, 0x7604u | (K << 4))); }
// same for the 128-byte-row table: lb2x = 2 * (table | lane*4)
template <int K> __device__ __forceinline__ uint32_t tab_half(uint32_t lb2x, uint32_t t) { return lds32(__byte_perm(t, lb2x, 0x7604u | (K << 4)) >> 1); }

// ---- GF(2^8) column arithmetic on packed words (row r of the column in byte r) -------------------
__device__ __forceinline__ uint32_t xtime4(uint32_t w) { return ((w & 0x7F7F7F7Fu) << 1) ^ (((w >> 7) & 0x01010101u) * 0x1Bu); }   // galois_mul2 :88-99, 4 bytes at once
__device__ __forceinline__ uint32_t mix_column(uint32_t w) {                   // :178-183: out_r = xtime(a_r ^ a_r+1) ^ a_r+1 ^ a_r+2 ^ a_r+3
    const uint32_t r1 = __byte_perm(w, 0u, 0x0321u), r2 = __byte_perm(w, 0u, 0x1032u), r3 = __byte_perm(w, 0u, 0x2103u);
    return xtime4(w ^ r1) ^ r1 ^ r2 ^ r3;
}
__device__ __forceinline__ uint32_t inv_mix_column(uint32_t w) {               // :172-177 pre-multiply, then the forward mix
    const uint32_t v = w ^ __byte_perm(w, 0u, 0x1032u);
    return mix_column(w ^ xtime4(xtime4(v)));
}

struct AesLaneBases { uint32_t lb0, lb1, lb2, lb3, sis2x; };

// SubWord(RotWord(w)) for the key schedule: bytes (S[w.b1], S[w.b2], S[w.b3], S[w.b0])
template <bool DEC> __device__ __forceinline__ uint32_t sub_rot_word(const AesLaneBases& L, uint32_t w) {
    if (DEC) {                                                  // S sits in bytes 1 and 3 of the (InvS, S, InvS, S) rows
        const uint32_t a = tab_half<1>(L.sis2x, w), b = tab_half<2>(L.sis2x, w), c = tab_half<3>(L.sis2x, w), d = tab_half<0>(L.sis2x, w);
        return __byte_perm(__byte_perm(a, b, 0x0051u), __byte_perm(c, d, 0x0051u), 0x5410u);
    }
    // S-box byte = byte 1 of TE0 = byte 2 of TE1 = byte 0 of TE2 ...
    return (tab<1>(L.lb2, w) & 0x000000FFu) | (tab<2>(L.lb0, w) & 0x0000FF00u) | (tab<3>(L.lb0, w) & 0x00FF0000u) | (tab<0>(L.lb1, w) & 0xFF000000u);
}
// forward key-schedule step (:214-221) and its inverse (:133-141), on the four key columns
template <bool DEC> __device__ __forceinline__ void key_next(const AesLaneBases& L, uint32_t (&k)[4], int rd) {
    k[0] ^= sub_rot_word<DEC>(L, k[3]) ^ (uint32_t)XMR_AES_RCON[rd];
    k[1] ^= k[0]; k[2] ^= k[1]; k[3] ^= k[2];
}
template <bool DEC> __device__ __forceinline__ void key_prev(const AesLaneBases& L, uint32_t (&k)[4], int rd) {
    k[3] ^= k[2]; k[2] ^= k[1]; k[1] ^= k[0];
    k[0] ^= sub_rot_word<DEC>(L, k[3]) ^ (uint32_t)XMR_AES_RCON[rd];
}

// one main-loop iteration without its AddRoundKey: encrypt = SubBytes+ShiftRows(+MixColumns), decrypt = InvShiftRows+InvSubBytes(+InvMixColumns)
template <bool DEC, bool LAST>
__device__ __forceinline__ void aes_round_cols(const AesLaneBases& L, const uint32_t (&t)[4], uint32_t (&n)[4]) {
    if (!DEC) {
        if (!LAST) {                                            // 4 table rows XORed
#pragma unroll
            for (int c = 0; c < 4; ++c)
                n[c] = tab<0>(L.lb0, t[c]) ^ tab<1>(L.lb1, t[(c + 1) & 3]) ^ tab<2>(L.lb2, t[(c + 2) & 3]) ^ tab<3>(L.lb3, t[(c + 3) & 3]);
        } else {                                                // round 9: no MixColumns (:168); S[x] sits in byte p of the table picked per position
#pragma unroll
            for (int c = 0; c < 4; ++c)
                n[c] = (tab<0>(L.lb2, t[c]) & 0x000000FFu) | (tab<1>(L.lb0, t[(c + 1) & 3]) & 0x0000FF00u) |
                       (tab<2>(L.lb0, t[(c + 2) & 3]) & 0x00FF0000u) | (tab<3>(L.lb1, t[(c + 3) & 3]) & 0xFF000000u);
        }
    } else {
        if (!LAST) {                                            // InvShiftRows: row r of column c comes from column c - r
#pragma unroll
            for (int c = 0; c < 4; ++c)
                n[c] = tab<0>(L.lb0, t[c]) ^ tab<1>(L.lb1, t[(c + 3) & 3]) ^ tab<2>(L.lb2, t[(c + 2) & 3]) ^ tab<3>(L.lb3, t[(c + 1) & 3]);
        } else {                                                // last iteration: plain InvSubBytes (byte 0 of the (InvS, S, InvS, S) rows)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const uint32_t a = tab_half<0>(L.sis2x, t[c]), b = tab_half<1>(L.sis2x, t[(c + 3) & 3]);
                const uint32_t d = tab_half<2>(L.sis2x, t[(c + 2) & 3]), e = tab_half<3>(L.sis2x, t[(c + 1) & 3]);
                n[c] = __byte_perm(__byte_perm(a, b, 0x0040u), __byte_perm(d, e, 0x0040u), 0x5410u);
            }
        }
    }
}

template <int NC>
__device__ __forceinline__ void aes_vote_store(const uint32_t (&c)[4], uint8_t* out, unsigned long long local,
                                               unsigned long long gunit, bool valid, int lane, uint32_t flags, Tally& tally) {
    const bool majority = flags & COAST_F_MAJORITY_D;
    uint32_t o[4], bad = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) { Voted v = vote_u32<NC, 1>(c[i], majority); o[i] = v.vote; bad += v.bad; }
    if (valid && Lanes<NC>::voter(lane)) {
        *reinterpret_cast<uint4*>(out + local * 16ull) = make_uint4(o[0], o[1], o[2], o[3]);
        tally.unit_exit<NC>(bad, 16u, flags, gunit);
    }
}

// The ten iterations of J blocks.  HOOKS = this warp has at least one block with a mid-round fault: the flip of block j is
// fbit[j] in column fcol[j] at the bottom of iteration frd[j].  PERKEY: k[j] is the block's running round key.
// ROLLED = keep the round loop a loop (PERKEY only: the round keys are then computed, not indexed): the rare hook path of the
// one-key kernels must stay SMALL -- a second fully unrolled copy of the rounds doubled the kernel to 82 KB and the two copies
// evicted each other from the instruction cache (r02 call 2b: +11 % instructions but +29 % time, issue rate 0.62 -> 0.55).
template <int J, bool DEC, bool PERKEY, bool HOOKS, bool ROLLED = false>
__device__ __forceinline__ void aes_rounds(const AesLaneBases& L, uint32_t (&s)[J][4], uint32_t (&k)[PERKEY ? J : 1][4], const uint32_t (&rk)[PERKEY ? 4 : 44],
                                           const uint32_t (&fbit)[J], const int (&frd)[J], const int (&fcol)[J]) {
    static_assert(!ROLLED || PERKEY, "a rolled round loop cannot index the register-resident round keys");
#pragma unroll (ROLLED ? 1 : 10)
    for (int rd = 0; rd < 10; ++rd) {
#pragma unroll
        for (int j = 0; j < J; ++j) {
            uint32_t n[4];
            if (rd < 9) aes_round_cols<DEC, false>(L, s[j], n); else aes_round_cols<DEC, true>(L, s[j], n);
            if (HOOKS) {                                        // the flip lands on state[] at the bottom of iteration rd
                uint32_t hit = frd[j] == rd ? fbit[j] : 0u;
                if (DEC && rd < 9) hit = inv_mix_column(hit);   // the kernel carries InvMixColumns(state) between decrypt iterations
#pragma unroll
                for (int c = 0; c < 4; ++c) n[c] ^= fcol[j] == c ? hit : 0u;
            }
            if (PERKEY) {
                if (!DEC) {
                    key_next<false>(L, k[j], rd);               // :214-221
#pragma unroll
                    for (int c = 0; c < 4; ++c) s[j][c] = n[c] ^ k[j][c];
                } else {
                    key_prev<true>(L, k[j], 9 - rd);            // :133-141 -> round key 9 - rd
#pragma unroll
                    for (int c = 0; c < 4; ++c) s[j][c] = n[c] ^ (rd < 9 ? inv_mix_column(k[j][c]) : k[j][c]);
                }
            } else {
                // encrypt: rk[4(rd+1)..] ; decrypt: rk[] already holds InvMixColumns(round key 9-rd) for rd < 9 and round key 0 last
#pragma unroll
                for (int c = 0; c < 4; ++c) s[j][c] = n[c] ^ rk[4 * (rd + 1) + c];
            }
        }
    }
}

// Hook path of the one-key kernels: the ten iterations as a ROLLED loop whose round keys come from a 176-byte copy in shared
// memory (broadcast reads).  Why this shape (profiles/r02_aes_injector_ablation_*.txt, DWC, 2^24 blocks, p = 2^-10):
//   second unrolled copy of the rounds (register keys) : 1.122 ms -- 35 KB more code; every execution evicts the fast path from the
//                                                         instruction cache of all 16 warps (issue rate 0.49)
//   rolled loop recomputing the key schedule            : 0.865 ms -- small, but 3x a normal tile per execution
//   rolled loop, keys from shared memory                : this one
template <int J, bool DEC>
__device__ __forceinline__ void aes_rounds_hooked(const AesLaneBases& L, uint32_t (&s)[J][4], uint32_t rk_saddr,
                                               const uint32_t (&fbit)[J], const int (&frd)[J], const int (&fcol)[J]) {
#pragma unroll 1
    for (int rd = 0; rd < 10; ++rd) {
        uint32_t kr[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) kr[c] = lds32(rk_saddr + 16u * (uint32_t)(rd + 1) + 4u * c);
#pragma unroll
        for (int j = 0; j < J; ++j) {
            uint32_t n[4];
            if (rd < 9) aes_round_cols<DEC, false>(L, s[j], n); else aes_round_cols<DEC, true>(L, s[j], n);
            uint32_t hit = frd[j] == rd ? fbit[j] : 0u;
            if (DEC && rd < 9) hit = inv_mix_column(hit);
#pragma unroll
            for (int c = 0; c < 4; ++c) s[j][c] = n[c] ^ (fcol[j] == c ? hit : 0u) ^ kr[c];
        }
    }
}

// the shared-memory tables of one direction (all threads of the CTA; the caller synchronises)
template <bool DEC>
__device__ __forceinline__ void aes_build_tables(uint8_t* smem_raw, uint32_t win, int tid) {
    uint32_t* t01 = reinterpret_cast<uint32_t*>(smem_raw + (AES_TAB01 - win));
    uint32_t* t23 = reinterpret_cast<uint32_t*>(smem_raw + (AES_TAB23 - win));
    for (int i = tid; i < 256 * 64; i += AES_THREADS) {
        uint32_t v;
        if (!DEC) v = XMR_AES_TE0[i >> 6];
        else v = inv_mix_column((uint32_t)XMR_AES_RSBOX[i >> 6]);   // TD0[x]: InvMixColumns of the column (InvS[x], 0, 0, 0) = (14, 9, 13, 11) . InvS[x]
        const bool hi = (i & 32) != 0;
        t01[i] = hi ? __byte_perm(v, 0u, 0x2103u) : v;                               // T1 = rotl8
        t23[i] = hi ? __byte_perm(v, 0u, 0x0321u) : __byte_perm(v, 0u, 0x1032u);     // T3 = rotl24 : T2 = rotl16
    }
    if (DEC) {
        uint32_t* sis = reinterpret_cast<uint32_t*>(smem_raw + (AES_SIS - win));
        for (int i = tid; i < 256 * 32; i += AES_THREADS) {
            const uint32_t is = XMR_AES_RSBOX[i >> 5], sb = XMR_AES_SBOX[i >> 5];
            sis[i] = is | (sb << 8) | (is << 16) | (sb << 24);
        }
    }
}
__device__ __forceinline__ AesLaneBases aes_lane_bases(int lane) {
    AesLaneBases L;
    L.lb0 = AES_TAB01 + 4u * lane; L.lb1 = AES_TAB01 + 128u + 4u * lane;
    L.lb2 = AES_TAB23 + 4u * lane; L.lb3 = AES_TAB23 + 128u + 4u * lane;
    L.sis2x = 2u * (AES_SIS + 4u * lane);
    return L;
}

// Deferred units of the one-key injector kernels.  A unit whose plan has a MID-ROUND flip is rare (p per block), and the code that
// applies such a flip is therefore cold; executing it inside the tile loop cost 1 000 - 3 500 SM cycles per hit in instruction
// fetch (profiles/r02_aes_injector_ablation_*.txt: the per-hit cost falls 9x when hits are 8x more frequent).  So the tile loop only
// QUEUES those units (per warp, in shared memory) and this pass -- run once per warp after its last tile -- does them: each group of
// NC adjacent lanes takes one queued unit, reloads its block, runs the ten iterations in a rolled one-block loop (round keys from
// shared memory) with the hook on the faulted replica's lane, votes and stores exactly as the tile loop would have.
constexpr int AES_QCAP = 96;                                  // entries per warp: 16 warps x 96 x 8 B = 12 KiB, placed after the ring below the first table window
template <int NC, bool DEC>
__device__ __noinline__ void aes_drain_deferred(const xmr_args& a, uint32_t rk_saddr, uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3,
                                                const uint32_t* q, uint32_t count, int lane) {
    constexpr int UPW = Lanes<NC>::kUnitsPerWarp;
    if (count == 0u) return;
    const AesLaneBases L = aes_lane_bases(lane);
    const int r = Lanes<NC>::replica(lane), g = Lanes<NC>::unit(lane);
    Tally tally(a);                                             // its own tally (flushed below): nothing of the caller's lives across this call
    __syncwarp();                                               // the voter lanes' queue writes are visible to the whole warp
    for (uint32_t base = 0; base < count; base += UPW) {
        const uint32_t idx = base + (uint32_t)g;
        const bool have = idx < count && (NC != 3 || lane < 30);
        const uint32_t lu = have ? q[2u * idx] : 0u, e = have ? q[2u * idx + 1u] : 0u;
        uint32_t x[1][4] = {{0u, 0u, 0u, 0u}}, fb[1] = {0u};
        int fr[1] = {-2}, fc[1] = {0};
        if (have) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(a.in) + (unsigned long long)lu * 16ull));
            x[0][0] = q.x ^ k0; x[0][1] = q.y ^ k1; x[0][2] = q.z ^ k2; x[0][3] = q.w ^ k3;
            if ((int)((e >> 29) & 3u) == r) {
                const uint32_t site = (e >> 5) & 0xFFFFFFu, i = (site - 16u) & 15u;
                fr[0] = (int)((site - 16u) >> 4); fc[0] = (int)(i >> 2); fb[0] = (1u << (e & 31u)) << (8u * (i & 3u));
            }
        }
        aes_rounds_hooked<1, DEC>(L, x, rk_saddr, fb, fr, fc);
        aes_vote_store<NC>(x[0], static_cast<uint8_t*>(a.out), (unsigned long long)lu, a.unit_base + lu, have, lane, a.flags, tally);
    }
    tally.flush(a.counters);
}

template <int NC, bool INJECT, bool DEC, bool PERKEY>
__device__ __forceinline__ void aes128_body(const xmr_args& a, const CUtensorMap* tmap) {
    constexpr int UPW = Lanes<NC>::kUnitsPerWarp;
    constexpr int J = AesGeom<NC>::J;
    constexpr int TROWS = AesGeom<NC>::TROWS;
    using Ring = AesRing<TROWS>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t win = smem_u32(smem_raw);                    // shared-window address of the dynamic region
    uint8_t* ring_mem = smem_raw + ((1024u - (win & 1023u)) & 1023u);
    Ring ring;
    ring.init(ring_mem, tmap, (a.mode & XMR_AES_ROWPACK_MASK) >> XMR_AES_ROWPACK_SHIFT);   // 16-byte blocks described as 64- or 256-byte rows
    // per-warp queue of deferred units (INJECT, one-key kernels): {unit, fault} pairs right after the ring, still below the tables
    constexpr uint32_t Q_OFF = (Ring::SMEM_BYTES + 127u) & ~127u;
    static_assert(Q_OFF + (uint32_t)AES_WARPS * AES_QCAP * 8u + 2048u + 1024u <= AES_TAB01, "ring + queues must end below the first table window");
    uint32_t* const q_mine = reinterpret_cast<uint32_t*>(ring_mem + Q_OFF) + (size_t)(threadIdx.x >> 5) * AES_QCAP * 2u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    aes_build_tables<DEC>(smem_raw, win, tid);
    __syncthreads();
    const AesLaneBases L = aes_lane_bases(lane);
    const int r = Lanes<NC>::replica(lane);
    const int u = Lanes<NC>::unit(lane);

    // One-key modes: every replica lane expands ITS OWN copy of the key (cloneGlobals: key[] is per-replica memory).
    //   encrypt: rk[4i..] = round key i.   decrypt: rk[0..3] = round key 10 (the first AddRoundKey, :127-129),
    //   rk[4(rd+1)..] = InvMixColumns(round key 9-rd) for rd < 9, rk[40..43] = round key 0.
    uint32_t rk[PERKEY ? 4 : 44];
    __shared__ uint32_t rk_shared[44];                          // INJECT && !PERKEY: the deferred pass reads its round keys here
    uint32_t q_count = 0u;                                      // entries in this warp's queue of deferred units (warp-uniform)
    if (!PERKEY) {
        uint32_t k[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            k[i] = (uint32_t)a.key[4 * i] | ((uint32_t)a.key[4 * i + 1] << 8) | ((uint32_t)a.key[4 * i + 2] << 16) | ((uint32_t)a.key[4 * i + 3] << 24);
        if (!DEC) {
#pragma unroll
            for (int c = 0; c < 4; ++c) rk[c] = k[c];
#pragma unroll
            for (int rd = 0; rd < 10; ++rd) {
                key_next<false>(L, k, rd);
#pragma unroll
                for (int c = 0; c < 4; ++c) rk[4 * (rd + 1) + c] = k[c];
            }
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) rk[40 + c] = k[c];      // round key 0
#pragma unroll
            for (int rd = 0; rd < 10; ++rd) {                   // :112-129; round key rd+1 is used by iteration 8-rd (rd < 9), round key 10 first
                key_next<true>(L, k, rd);
#pragma unroll
                for (int c = 0; c < 4; ++c) rk[rd < 9 ? 4 * (9 - rd) + c : c] = rd < 9 ? inv_mix_column(k[c]) : k[c];
            }
        }
    }

    if (INJECT && !PERKEY) {
        if (tid == 0) {
#pragma unroll
            for (int i = 0; i < 44; ++i) rk_shared[i] = rk[i];
        }
        __syncthreads();
    }
    const uint32_t n_tiles = a.n_tiles;
    uint32_t tile = blockIdx.x;
    if (tid == 0) {                                             // prologue: AES_STAGES - 1 tiles in flight
#pragma unroll
        for (uint32_t i = 0; i + 1u < (uint32_t)AES_STAGES; ++i)
            if (tile + i * gridDim.x < n_tiles) ring.issue(i, tile + i * gridDim.x);
    }
    Tally tally(a);
    uint32_t it = 0;
    for (; tile < n_tiles; tile += gridDim.x, ++it) {
        const uint8_t* base = ring.wait_full(it);
        uint32_t s[J][4];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            uint4 q = *reinterpret_cast<const uint4*>(base + ((warp * J + j) * UPW + u) * 16);
            s[j][0] = q.x; s[j][1] = q.y; s[j][2] = q.z; s[j][3] = q.w;
        }
        ring.release(it, lane);
        if (tid == 0) {                                         // refill: tile it + STAGES - 1 goes where tile it - 1 was
            const uint32_t ahead = tile + (uint32_t)(AES_STAGES - 1) * gridDim.x;
            if (ahead < n_tiles) {
                if (it >= 1u) ring.wait_empty(it - 1u);
                ring.issue(it + (uint32_t)(AES_STAGES - 1), ahead);
            }
        }

        unsigned long long local[J];
        bool valid[J];
        uint32_t k[PERKEY ? J : 1][4];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            local[j] = (unsigned long long)tile * TROWS + (unsigned)((warp * J + j) * UPW + u);
            valid[j] = local[j] < a.n_units;
            if (PERKEY) {
                uint4 kq = make_uint4(0u, 0u, 0u, 0u);
                if (valid[j]) kq = __ldg(reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(a.aux) + local[j] * 16ull));
                k[j][0] = kq.x; k[j][1] = kq.y; k[j][2] = kq.z; k[j][3] = kq.w;
            }
        }
        // fault of block j as masks: column word fcol[j], shifted bit fbit[j], applied at the bottom of iteration frd[j]
        // (frd = -1: the replica's input copy, before the first AddRoundKey; -2: none)
        uint32_t fbit[J]; int frd[J], fcol[J];
        bool hooks = false;
        uint32_t defer = 0u;                                    // one-key kernels: bit j = unit of block j has a mid-round flip -> deferred (below)
#pragma unroll
        for (int j = 0; j < J; ++j) { fbit[j] = 0u; frd[j] = -2; fcol[j] = 0; }
        if (INJECT) {
            // The unit's Philox draw is evaluated ONCE, by one lane, with every lane of the warp busy in the same instruction:
            // in pass t, replica lane r evaluates block j = t * NC + r of its unit (different lanes, different blocks -- no
            // divergence), so a warp spends ceil(J / NC) evaluations per lane instead of J (r02 call 2: the per-j `if (r == j % NC)`
            // form diverged and cost all J; r01 evaluated every block on every replica lane).
            constexpr int PASSES = (J + NC - 1) / NC;
            uint32_t packed[PASSES];
#pragma unroll
            for (int t = 0; t < PASSES; ++t) {
                const int jt = t * NC + r;                       // this lane's block in pass t
                const bool mine = jt < J;
                const unsigned long long lo = (unsigned long long)tile * TROWS + (unsigned)((warp * J + (mine ? jt : 0)) * UPW + u);
                const bool ok = mine && lo < a.n_units;
                Fault f = fault_for_unit(a, NC, ok ? lo : 0ull, [](uint32_t) { return 8u; });
                packed[t] = (f.active && ok) ? (0x80000000u | (f.replica << 29) | (f.site << 5) | f.bit) : 0u;
            }
            bool mid = false;
            uint32_t any_packed = 0u;
#pragma unroll
            for (int t = 0; t < PASSES; ++t) any_packed |= packed[t];
            if (__any_sync(0xFFFFFFFFu, any_packed != 0u)) {    // 94 % of warp-tiles at p = 2^-10 have no hit at all: skip the distribution
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    const uint32_t e = NC == 1 ? packed[j] : __shfl_sync(0xFFFFFFFFu, packed[j / NC], u * NC + j % NC);
                    const uint32_t site = (e >> 5) & 0xFFFFFFu, bit = e & 31u;
                    const bool hit = (e & 0x80000000u) != 0u;
                    if (hit && Lanes<NC>::voter(lane)) tally.injected++;
                    if (!PERKEY) {
                        // ONE-KEY KERNELS: a unit with a MID-ROUND flip is not finished here.  All its replica lanes skip the vote/store
                        // of that block; the voter lane queues (unit, fault) for the pass after the tile loop (aes_drain_deferred).
                        const bool dq = hit && site >= 16u;
                        if (dq) defer |= 1u << j;
                        const uint32_t pushers = __ballot_sync(0xFFFFFFFFu, dq && Lanes<NC>::voter(lane));
                        if (dq && Lanes<NC>::voter(lane)) {
                            const uint32_t pos = q_count + __popc(pushers & ((1u << lane) - 1u));
                            if (pos < (uint32_t)AES_QCAP) { q_mine[2u * pos] = (uint32_t)local[j]; q_mine[2u * pos + 1u] = e; }
                        }
                        q_count += __popc(pushers);             // warp-uniform
                    }
                    if (hit && (PERKEY || site < 16u) && (int)((e >> 29) & 3u) == r) {
                        const uint32_t i = site < 16u ? site : ((site - 16u) & 15u);
                        frd[j] = site < 16u ? -1 : (int)((site - 16u) >> 4);
                        fcol[j] = (int)(i >> 2);
                        fbit[j] = (1u << bit) << (8u * (i & 3u));
                        if (frd[j] < 0) {                       // the replica's private copy of its input
#pragma unroll
                            for (int c = 0; c < 4; ++c) s[j][c] ^= fcol[j] == c ? fbit[j] : 0u;
                        } else mid = true;
                    }
                }
                hooks = __any_sync(0xFFFFFFFFu, mid);           // per-unit-key kernels: a warp without a mid-round hit runs the plain rounds
            }
        }
#pragma unroll
        for (int j = 0; j < J; ++j) {
            if (PERKEY && DEC) {
#pragma unroll
                for (int rd = 0; rd < 10; ++rd) key_next<true>(L, k[j], rd);      // :112-126: run the schedule to the last round key
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) s[j][c] ^= PERKEY ? k[j][c] : rk[c];      // first half of :143-146 / :127-129
        }
        if constexpr (PERKEY) {
            if (INJECT && hooks) aes_rounds<J, DEC, true, true, true>(L, s, k, rk, fbit, frd, fcol);     // per-unit keys: rolled, keys recomputed
            else aes_rounds<J, DEC, true, false>(L, s, k, rk, fbit, frd, fcol);
        } else {
            aes_rounds<J, DEC, false, false>(L, s, k, rk, fbit, frd, fcol);
        }
#pragma unroll
        for (int j = 0; j < J; ++j) {
            aes_vote_store<NC>(s[j], static_cast<uint8_t*>(a.out), local[j], a.unit_base + local[j], valid[j] && !((defer >> j) & 1u), lane, a.flags, tally);
            if (PERKEY && (a.mode & 4u) && valid[j] && Lanes<NC>::voter(lane))       // COAST_AES_KEY_WRITEBACK: replica 0's mutated key[]
                *reinterpret_cast<uint4*>(static_cast<uint8_t*>(const_cast<void*>(a.aux)) + local[j] * 16ull) = make_uint4(k[j][0], k[j][1], k[j][2], k[j][3]);
        }
        if (INJECT && !PERKEY && q_count > (uint32_t)(AES_QCAP - J * UPW)) {        // the next tile might not fit: drain now (rare)
            aes_drain_deferred<NC, DEC>(a, smem_u32(rk_shared), rk[0], rk[1], rk[2], rk[3], q_mine, q_count, lane);
            q_count = 0u;
        }
    }
    if (INJECT && !PERKEY) aes_drain_deferred<NC, DEC>(a, smem_u32(rk_shared), rk[0], rk[1], rk[2], rk[3], q_mine, q_count, lane);
    tally.flush(a.counters);
}

// ---------------------------------------------------------------------------------------------
// CHStone `aes` (tests/chstone/aes/aes_enc.c:66-134, aes_dec.c:66-140, aes_func.c, aes_key.c; type 128128): the same
// cipher with one byte per `int`.  Unit = one block: 16 ints in (64 bytes), 16 ints out; the key (16 ints per unit in
// d_aux, or the 16 bytes of the descriptor) is expanded on the fly per replica and never written back (KeySchedule fills
// word[][], aes_key.c:129-163, the key itself is untouched).  SoR exit = the 16 `int` elements of statemt (compared one
// by one, aes_enc.c:130-131): 16 votes.  Same rounds, tables and fault hooks as the TI kernel; a fault site is
// "statemt[i] right after a round-key addition", which is where the TI enumeration puts it too (header).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack4(uint4 q) { return (q.x & 0xFFu) | ((q.y & 0xFFu) << 8) | ((q.z & 0xFFu) << 16) | ((q.w & 0xFFu) << 24); }
__device__ __forceinline__ uint4 unpack4(uint32_t w) { return make_uint4(w & 0xFFu, (w >> 8) & 0xFFu, (w >> 16) & 0xFFu, w >> 24); }

template <int NC, bool INJECT, bool DEC>
__device__ __forceinline__ void chstone_aes_body(const xmr_args& a) {
    constexpr int UPW = Lanes<NC>::kUnitsPerWarp;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    const uint32_t win = smem_u32(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31;
    aes_build_tables<DEC>(smem_raw, win, tid);
    __syncthreads();
    const AesLaneBases L = aes_lane_bases(lane);
    const int r = Lanes<NC>::replica(lane);
    const unsigned long long gwarp = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    const unsigned long long n_wtiles = (a.n_units + UPW - 1) / UPW;
    const bool per_unit = a.mode & 2u;
    const bool majority = a.flags & COAST_F_MAJORITY_D;
    const uint32_t rk_unused[4] = {0u, 0u, 0u, 0u};
    Tally tally(a);
    for (unsigned long long wt = gwarp; wt < n_wtiles; wt += nwarps) {
        const unsigned long long local = wt * UPW + Lanes<NC>::unit(lane);
        const bool valid = local < a.n_units;
        const unsigned long long ld = valid ? local : 0ull;
        uint32_t s[1][4], k[1][4];
        const uint4* ip = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(a.in) + ld * 64ull);
#pragma unroll
        for (int c = 0; c < 4; ++c) s[0][c] = pack4(__ldg(ip + c));
        if (per_unit) {
            const uint4* kp = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(a.aux) + ld * 64ull);
#pragma unroll
            for (int c = 0; c < 4; ++c) k[0][c] = pack4(__ldg(kp + c));
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c)
                k[0][c] = (uint32_t)a.key[4 * c] | ((uint32_t)a.key[4 * c + 1] << 8) | ((uint32_t)a.key[4 * c + 2] << 16) | ((uint32_t)a.key[4 * c + 3] << 24);
        }
        uint32_t fbit[1] = {0u}; int frd[1] = {-2}, fcol[1] = {0};
        bool hooks = false;
        if (INJECT) {
            Fault f = fault_for_unit(a, NC, ld, [](uint32_t) { return 8u; });
            bool mid = false;
            if (f.active && valid) {
                if (Lanes<NC>::voter(lane)) tally.injected++;
                if ((int)f.replica == r) {
                    const uint32_t i = f.site < 16u ? f.site : ((f.site - 16u) & 15u);
                    frd[0] = f.site < 16u ? -1 : (int)((f.site - 16u) >> 4);
                    fcol[0] = (int)(i >> 2);
                    fbit[0] = (1u << f.bit) << (8u * (i & 3u));
                    if (frd[0] < 0) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) s[0][c] ^= fcol[0] == c ? fbit[0] : 0u;
                    } else mid = true;
                }
            }
            hooks = __any_sync(0xFFFFFFFFu, mid);
        }
        if (DEC) {
#pragma unroll
            for (int rd = 0; rd < 10; ++rd) key_next<true>(L, k[0], rd);          // word[][40..43]: the last round key (aes_dec.c:115)
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) s[0][c] ^= k[0][c];                           // AddRoundKey(0) / AddRoundKey(10)
        if (INJECT && hooks) aes_rounds<1, DEC, true, true, true>(L, s, k, rk_unused, fbit, frd, fcol);
        else aes_rounds<1, DEC, true, false>(L, s, k, rk_unused, fbit, frd, fcol);
        uint32_t o[4], bad = 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) { Voted v = vote_u32<NC, 1>(s[0][c], majority); o[c] = v.vote; bad += v.bad; }   // one byte per int: 16 element votes
        if (valid && Lanes<NC>::voter(lane)) {
            uint4* op = reinterpret_cast<uint4*>(static_cast<uint8_t*>(a.out) + local * 64ull);
#pragma unroll
            for (int c = 0; c < 4; ++c) op[c] = unpack4(o[c]);
            tally.unit_exit<NC>(bad, 16u, a.flags, a.unit_base + local);
        }
    }
    tally.flush(a.counters);
}

}  // namespace xmr

#define XMR_AES_KERNEL(NAME, NC, INJ, DEC, PERKEY)                                                       \
    extern "C" __global__ void __launch_bounds__(xmr::AES_THREADS, 1)                                    \
    xmr_aes128_##NAME##_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a, const __grid_constant__ CUtensorMap tmap) { \
        xmr::aes128_body<NC, INJ != 0, DEC, PERKEY>(a, &tmap);                                           \
    }
#define XMR_AES_ALL(NC, INJ) \
    XMR_AES_KERNEL(enc, NC, INJ, false, false) XMR_AES_KERNEL(dec, NC, INJ, true, false) \
    XMR_AES_KERNEL(enck, NC, INJ, false, true) XMR_AES_KERNEL(deck, NC, INJ, true, true)
XMR_AES_ALL(1, 0) XMR_AES_ALL(2, 0) XMR_AES_ALL(3, 0)
XMR_AES_ALL(1, 1) XMR_AES_ALL(2, 1) XMR_AES_ALL(3, 1)
#define XMR_CHAES_KERNEL(NAME, NC, INJ, DEC)                                                             \
    extern "C" __global__ void __launch_bounds__(xmr::AES_THREADS, 1)                                    \
    xmr_chaes_##NAME##_nc##NC##_inj##INJ(const __grid_constant__ xmr_args a) { xmr::chstone_aes_body<NC, INJ != 0, DEC>(a); }
#define XMR_CHAES_ALL(NC, INJ) XMR_CHAES_KERNEL(enc, NC, INJ, false) XMR_CHAES_KERNEL(dec, NC, INJ, true)
XMR_CHAES_ALL(1, 0) XMR_CHAES_ALL(2, 0) XMR_CHAES_ALL(3, 0)
XMR_CHAES_ALL(1, 1) XMR_CHAES_ALL(2, 1) XMR_CHAES_ALL(3, 1)
