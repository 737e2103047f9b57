/*
 * xmr_args.h -- kernel argument block shared by the host runtime (coast_rt.c, plain C)
 * and the sm_100a kernels (coast_kernels.cu).  Plain C layout, no CUDA types.
 */
#ifndef XMR_ARGS_H_
#define XMR_ARGS_H_

typedef struct xmr_args {
    const void* in;
    void* out;
    const void* aux;
    unsigned long long n_units;
    unsigned long long unit_base;
    unsigned long long* counters;     /* XMR_CTR_* slots, device memory            */
    const unsigned int* plan_table;   /* COAST_PLAN_TABLE: one u32 per local unit  */
    unsigned char* status;            /* optional: per-unit count of disagreeing votes (saturating u8) */
    unsigned int unit_bytes;
    unsigned int flags;               /* COAST_F_*                                  */
    unsigned int mode;                /* COAST_AES_*                                */
    unsigned int M, N, K;
    unsigned int plan_mode, seed_lo, seed_hi, threshold;
    unsigned int n_sites;
    unsigned int n_tiles;             /* TMA-tiled kernels: ceil(n_units / units-per-tile) */
    unsigned char key[16];
} xmr_args;

/* internal flag (set by the host in xmr_args.flags, never by callers): in-loop store votes are in effect (coast_rt.h) */
#define XMR_F_STORE_VOTES 0x8000u
/* AES: bits 8..11 of xmr_args.mode = log2 of the blocks per tensor-map row (the host describes the dense 16-byte blocks as
 * 64- or 256-byte rows when the count allows) */
#define XMR_AES_ROWPACK_SHIFT 8u
#define XMR_AES_ROWPACK_MASK  (15u << XMR_AES_ROWPACK_SHIFT)

/* counter slots (mirror coast_stats) */
#define XMR_CTR_ERRORS   0
#define XMR_CTR_DWC      1
#define XMR_CTR_SYNCS    2
#define XMR_CTR_INJECTED 3
#define XMR_CTR_FIRST    4
#define XMR_CTR_COUNT    5

/* tile geometry of the TMA-staged kernels: CTA = 8 warps, each warp owns 32/NC units */
#define XMR_CTA_THREADS 256
#define XMR_WARPS       8
#define XMR_STAGES      2

#endif
