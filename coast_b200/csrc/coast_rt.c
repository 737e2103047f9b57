/*
 * coast_rt.c -- host side of libcoast_rt.so (plain C over the CUDA DRIVER API).
 *
 * Replaces, at run time, what byuccl/coast does at compile time:
 *   projects/dataflowProtection (run(M, numClones), dataflowProtection.cpp:63-164),
 *   projects/TMR (TMR.cpp:29-36) and projects/DWC (DWC.cpp:29-36)
 * by launching a hand-written sm_100a kernel in which every live value of the protected
 * region is computed by num_clones replicas and voted at the SoR exit.
 *
 * libcuda.so.1 is bound lazily with dlopen() so that this library LOADS without a GPU
 * (the CPU CI box) -- every compute entry point then returns COAST_ERR_NO_DRIVER.  There
 * is deliberately NO CPU implementation of the workloads in this file.
 */
#define _GNU_SOURCE
#include "../../include/coast_rt.h"
#include "xmr_args.h"

#include <cuda.h>
#include <ctype.h>
#include <dlfcn.h>
#include <sched.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/syscall.h>
#include <unistd.h>

extern const unsigned char coast_kernels_cubin[];   /* generated: bin2c of coast_kernels.cubin */

/* ------------------------------------------------------------------ */
/* the reference's run-time symbols                                     */
/* ------------------------------------------------------------------ */
__attribute__((weak)) uint32_t TMR_ERROR_CNT = 0;    /* synchronization.cpp:269-291 */
__attribute__((weak)) uint64_t __SYNC_COUNT = 0;     /* synchronization.cpp:103-121 */
__attribute__((weak)) void FAULT_DETECTED_DWC(void) { /* synchronization.cpp:1251-1266: default handler = abort() */
    fprintf(stderr, "coast_rt: DWC mismatch detected -> FAULT_DETECTED_DWC -> abort()\n");
    abort();
}

/* ------------------------------------------------------------------ */
/* driver API binding                                                   */
/* ------------------------------------------------------------------ */
#define DRV_FUNCS(X)                                                                                         \
    X(cuInit, (unsigned int))                                                                                \
    X(cuDeviceGet, (CUdevice*, int))                                                                         \
    X(cuDeviceGetAttribute, (int*, CUdevice_attribute, CUdevice))                                            \
    X(cuDeviceGetPCIBusId, (char*, int, CUdevice))                                                           \
    X(cuPointerGetAttribute, (void*, CUpointer_attribute, CUdeviceptr))                                      \
    X(cuDevicePrimaryCtxRetain, (CUcontext*, CUdevice))                                                      \
    X(cuDevicePrimaryCtxRelease_v2, (CUdevice))                                                              \
    X(cuCtxSetCurrent, (CUcontext))                                                                          \
    X(cuCtxGetCurrent, (CUcontext*))                                                                         \
    X(cuModuleLoadData, (CUmodule*, const void*))                                                            \
    X(cuModuleUnload, (CUmodule))                                                                            \
    X(cuModuleGetFunction, (CUfunction*, CUmodule, const char*))                                             \
    X(cuFuncSetAttribute, (CUfunction, CUfunction_attribute, int))                                           \
    X(cuOccupancyMaxActiveBlocksPerMultiprocessor, (int*, CUfunction, int, size_t))                          \
    X(cuLaunchKernel, (CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned,     \
                       CUstream, void**, void**))                                                            \
    X(cuMemAlloc_v2, (CUdeviceptr*, size_t))                                                                 \
    X(cuMemFree_v2, (CUdeviceptr))                                                                           \
    X(cuMemPoolCreate, (CUmemoryPool*, const CUmemPoolProps*))                                               \
    X(cuMemPoolDestroy, (CUmemoryPool))                                                                      \
    X(cuMemPoolSetAttribute, (CUmemoryPool, CUmemPool_attribute, void*))                                     \
    X(cuMemAllocFromPoolAsync, (CUdeviceptr*, size_t, CUmemoryPool, CUstream))                               \
    X(cuMemFreeAsync, (CUdeviceptr, CUstream))                                                               \
    X(cuMemcpyHtoDAsync_v2, (CUdeviceptr, const void*, size_t, CUstream))                                    \
    X(cuMemcpyDtoHAsync_v2, (void*, CUdeviceptr, size_t, CUstream))                                          \
    X(cuMemcpyDtoDAsync_v2, (CUdeviceptr, CUdeviceptr, size_t, CUstream))                                    \
    X(cuMemsetD8Async, (CUdeviceptr, unsigned char, size_t, CUstream))                                       \
    X(cuMemHostAlloc, (void**, size_t, unsigned int))                                                        \
    X(cuMemFreeHost, (void*))                                                                                \
    X(cuStreamCreate, (CUstream*, unsigned int))                                                             \
    X(cuStreamDestroy_v2, (CUstream))                                                                        \
    X(cuStreamSynchronize, (CUstream))                                                                       \
    X(cuEventCreate, (CUevent*, unsigned int))                                                               \
    X(cuEventRecord, (CUevent, CUstream))                                                                    \
    X(cuEventDestroy_v2, (CUevent))                                                                          \
    X(cuStreamWaitEvent, (CUstream, CUevent, unsigned int))                                                  \
    X(cuGetErrorString, (CUresult, const char**))                                                            \
    X(cuIpcGetMemHandle, (CUipcMemHandle*, CUdeviceptr))                                                     \
    X(cuIpcOpenMemHandle_v2, (CUdeviceptr*, CUipcMemHandle, unsigned int))                                   \
    X(cuIpcCloseMemHandle, (CUdeviceptr))                                                                    \
    X(cuTensorMapEncodeTiled, (CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,      \
                               const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, \
                               CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill))

#define X(name, args) static CUresult(CUDAAPI* p_##name) args;
DRV_FUNCS(X)
#undef X

#define MAX_FN 128
static struct {
    int inited;
    void* libcuda;
    int device;
    CUdevice dev;
    CUcontext ctx;
    CUmodule mod;
    int sm_count;
    CUdeviceptr counters;            /* XMR_CTR_COUNT x u64 */
    CUdeviceptr peer_counters;       /* coast_counters_attach(): ANOTHER GPU's counter block, mapped over NVLink (0: not attached) */
    uint64_t* h_counters;            /* pinned mirror */
    struct { char name[64]; CUfunction fn; int ctas_per_sm; unsigned smem; } fns[MAX_FN];
    int n_fns;
    char err[512];
    /* protection mode of the four reference entry points (coast_set_opt_passes / COAST_OPT_PASSES) */
    uint32_t def_nc, def_flags; int def_set;
    /* coast_run_host scratch: 3 slots */
    CUstream hs[3]; CUdeviceptr h_in[3], h_out[3], h_aux[3]; size_t h_in_cap[3], h_out_cap[3], h_aux_cap[3];
    /* stream-ordered scratch (the replicas' private arrays of xmr_qsort.cuh): any number of streams may launch at once */
    CUmemoryPool pool;
    CUdeviceptr h_stat[3]; size_t h_stat_cap[3];     /* per-slot d_status staging of coast_run_host */
    CUdeviceptr h_b; size_t h_b_cap; CUevent ev_b;   /* matmul host call: the replicated operand B and "B has landed" */
    int numa_node;                   /* NUMA node the process was bound to by coast_init (-1: not bound) */
    int busy;                        /* one host thread at a time (the reference is single-threaded); others fail loudly */
    /* tensor maps of the row-tiled kernels, keyed by (base, row bytes, rows, box rows, swizzle): coast_run_host re-encodes the
     * same few maps every call */
    struct { const void* base; uint32_t row_bytes, box_rows; uint64_t rows; int swz; CUtensorMap map; } tmaps[16];
    int n_tmaps, tmap_next;
    unsigned warned_store_votes;     /* one warning per kernel and process */
    const char* last_host_path;      /* "staged" | "hybrid" | "zerocopy" | "row-blocks" | "one-shot": what the last coast_run_host did */
} G;

/* Single-caller guard.  The reference's emitted code is single-threaded (plain load/add/store on its counters,
 * synchronization.cpp:1428-1431) and so is this runtime: one counter block, one set of host-call slots.  A second host
 * thread entering while a call is in progress gets COAST_ERR_BUSY instead of a silent race. */
static int enter(void);
static void leave(void) { __atomic_store_n(&G.busy, 0, __ATOMIC_RELEASE); }

static int fail(int code, const char* fmt, ...) {
    va_list ap; va_start(ap, fmt);
    vsnprintf(G.err, sizeof G.err, fmt, ap);
    va_end(ap);
    return code;
}
static int enter(void) {
    if (__atomic_exchange_n(&G.busy, 1, __ATOMIC_ACQUIRE)) {
        /* do not touch G.err: the call in progress owns it */
        return COAST_ERR_BUSY;
    }
    return COAST_OK;
}
#define ENTER() do { int e_ = enter(); if (e_) return e_; } while (0)
#define LEAVE(rc) do { int l_ = (rc); leave(); return l_; } while (0)
static int drv_fail(CUresult r, const char* what) {
    const char* s = NULL;
    if (p_cuGetErrorString) p_cuGetErrorString(r, &s);
    return fail(-(int)r, "%s: CUDA error %d (%s)", what, (int)r, s ? s : "?");
}
#define DRV(call) do { CUresult r_ = (call); if (r_ != CUDA_SUCCESS) return drv_fail(r_, #call); } while (0)

const char* coast_last_error(void) { return G.err; }
const char* coast_version(void) { return "coast_rt 0.1 (sm_100a)"; }

static int bind_driver(void) {
    if (G.libcuda) return COAST_OK;
    void* h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libcuda.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(COAST_ERR_NO_DRIVER, "libcuda.so.1 not found (%s): no GPU driver on this machine; "
                                              "libcoast_rt has no CPU fallback", dlerror());
#define X(name, args)                                                                 \
    *(void**)(&p_##name) = dlsym(h, #name);                                           \
    if (!p_##name) { dlclose(h); return fail(COAST_ERR_NO_DRIVER, "libcuda lacks %s", #name); }
    DRV_FUNCS(X)
#undef X
    G.libcuda = h;
    return COAST_OK;
}


/* ------------------------------------------------------------------ */
/* NUMA placement                                                        */
/* ------------------------------------------------------------------ */
/* The host-call path (coast_run_host) is PCIe-bound; on a two-socket box a process that runs -- and first-touches its
 * pinned buffers -- on the socket the GPU is NOT attached to loses up to half of the copy bandwidth (measured r01: 1.69 vs
 * 3.16 ms per 96 MiB step on two boxes).  coast_init() therefore moves the calling thread (threads it creates later inherit
 * it) onto the CPUs of the GPU's NUMA node and makes that node the preferred one for its memory.  Plain syscalls, no
 * libnuma.  COAST_NUMA_BIND=0 leaves the process alone.  Best effort: any failure leaves things as they were. */
#ifndef MPOL_PREFERRED
#define MPOL_PREFERRED 1
#endif
static int parse_cpulist(const char* s, cpu_set_t* set) {
    int n = 0;
    CPU_ZERO(set);
    while (*s) {
        while (*s == ',' || isspace((unsigned char)*s)) ++s;
        if (!isdigit((unsigned char)*s)) break;
        char* e; long a = strtol(s, &e, 10), b = a;
        if (*e == '-') b = strtol(e + 1, &e, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET((int)c, set); ++n; }
        s = e;
    }
    return n;
}
static void numa_bind_to_gpu(void) {
    G.numa_node = -1;
    const char* env = getenv("COAST_NUMA_BIND");
    if (env && !strcmp(env, "0")) return;
    char bdf[32] = {0}, path[128], buf[4096];
    if (p_cuDeviceGetPCIBusId(bdf, (int)sizeof bdf - 1, G.dev) != CUDA_SUCCESS) return;
    for (char* c = bdf; *c; ++c) *c = (char)tolower((unsigned char)*c);
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bdf);
    FILE* f = fopen(path, "r"); if (!f) return;
    int node = -1; if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f);
    if (node < 0 || node >= 1024) return;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r"); if (!f) return;
    size_t got = fread(buf, 1, sizeof buf - 1, f); fclose(f); buf[got] = 0;
    cpu_set_t want, cur, both;
    if (!parse_cpulist(buf, &want)) return;
    if (sched_getaffinity(0, sizeof cur, &cur)) return;
    CPU_AND(&both, &want, &cur);                       /* never widen a cpuset the launcher (cgroup, taskset) imposed */
    if (!CPU_COUNT(&both)) return;
    if (sched_setaffinity(0, sizeof both, &both)) return;
    unsigned long mask[16]; memset(mask, 0, sizeof mask);
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    syscall(SYS_set_mempolicy, MPOL_PREFERRED, mask, (unsigned long)(8 * sizeof mask));   /* a refusal only costs locality */
    G.numa_node = node;
}
int coast_numa_node(void) { return G.inited ? G.numa_node : -1; }

static int ensure_ctx(void) {
    if (!G.inited) return fail(COAST_ERR_NOT_INIT, "coast_init() has not been called");
    CUcontext cur = NULL;
    p_cuCtxGetCurrent(&cur);
    if (cur != G.ctx) DRV(p_cuCtxSetCurrent(G.ctx));
    return COAST_OK;
}

static int get_fn_b(const char* name, unsigned smem, int block, CUfunction* fn, int* ctas_per_sm) {
    for (int i = 0; i < G.n_fns; ++i)
        if (!strcmp(G.fns[i].name, name) && G.fns[i].smem == smem) { *fn = G.fns[i].fn; if (ctas_per_sm) *ctas_per_sm = G.fns[i].ctas_per_sm; return COAST_OK; }
    CUfunction f = NULL;
    CUresult r = p_cuModuleGetFunction(&f, G.mod, name);
    if (r != CUDA_SUCCESS) return drv_fail(r, name);
    if (smem > 48 * 1024) DRV(p_cuFuncSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem));
    int occ = 1;
    DRV(p_cuOccupancyMaxActiveBlocksPerMultiprocessor(&occ, f, block, smem));
    if (occ < 1) occ = 1;
    if (G.n_fns < MAX_FN) {
        snprintf(G.fns[G.n_fns].name, sizeof G.fns[0].name, "%s", name);
        G.fns[G.n_fns].fn = f; G.fns[G.n_fns].ctas_per_sm = occ; G.fns[G.n_fns].smem = smem;
        G.n_fns++;
    }
    *fn = f; if (ctas_per_sm) *ctas_per_sm = occ;
    return COAST_OK;
}

static int get_fn(const char* name, unsigned smem, CUfunction* fn, int* ctas_per_sm) {
    return get_fn_b(name, smem, XMR_CTA_THREADS, fn, ctas_per_sm);
}

static int launch_small(const char* name, unsigned grid, unsigned block, void** params, CUstream s) {
    CUfunction f; int rc = get_fn(name, 0, &f, NULL);
    if (rc) return rc;
    DRV(p_cuLaunchKernel(f, grid, 1, 1, block, 1, 1, 0, s, params, NULL));
    return COAST_OK;
}

static int stats_reset_impl(void* stream) {
    int rc = ensure_ctx(); if (rc) return rc;
    void* params[] = { &G.counters };
    return launch_small("xmr_counters_reset", 1, 32, params, (CUstream)stream);
}
int coast_stats_reset(void* stream) { ENTER(); LEAVE(stats_reset_impl(stream)); }

/* COAST_REPORT_COUNTERS=1: print the reference's two run-time symbols when the process exits -- what a debugger would read
 * out of a board (passes.rst "Error Logging"); the unchanged tests never print them */
static void report_counters(void) {
    fprintf(stderr, "coast_rt: TMR_ERROR_CNT=%u __SYNC_COUNT=%llu\n", TMR_ERROR_CNT, (unsigned long long)__SYNC_COUNT);
}

static int init_impl(int device) {
    if (G.inited) {
        if (device == G.device) return ensure_ctx();
        return fail(COAST_ERR_BAD_ARG, "coast_rt already initialised on device %d", G.device);
    }
    int rc = bind_driver(); if (rc) return rc;
    CUresult r = p_cuInit(0);
    if (r != CUDA_SUCCESS) { drv_fail(r, "cuInit"); return COAST_ERR_NO_DRIVER; }
    DRV(p_cuDeviceGet(&G.dev, device));
    DRV(p_cuDevicePrimaryCtxRetain(&G.ctx, G.dev));      /* shared with the CUDA runtime / torch */
    DRV(p_cuCtxSetCurrent(G.ctx));
    int major = 0, minor = 0;
    p_cuDeviceGetAttribute(&major, CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MAJOR, G.dev);
    p_cuDeviceGetAttribute(&minor, CU_DEVICE_ATTRIBUTE_COMPUTE_CAPABILITY_MINOR, G.dev);
    if (major != 10) {
        p_cuDevicePrimaryCtxRelease_v2(G.dev);
        return fail(COAST_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library carries sm_100a code only", device, major, minor);
    }
    p_cuDeviceGetAttribute(&G.sm_count, CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT, G.dev);
    numa_bind_to_gpu();
    r = p_cuModuleLoadData(&G.mod, coast_kernels_cubin);
    if (r != CUDA_SUCCESS) { p_cuDevicePrimaryCtxRelease_v2(G.dev); return drv_fail(r, "cuModuleLoadData(sm_100a cubin)"); }
    DRV(p_cuMemAlloc_v2(&G.counters, XMR_CTR_COUNT * sizeof(uint64_t)));
    {
        CUmemPoolProps pp; memset(&pp, 0, sizeof pp);
        pp.allocType = CU_MEM_ALLOCATION_TYPE_PINNED;
        pp.location.type = CU_MEM_LOCATION_TYPE_DEVICE; pp.location.id = (int)G.dev;
        DRV(p_cuMemPoolCreate(&G.pool, &pp));
        cuuint64_t keep = ~(cuuint64_t)0;                  /* keep freed scratch cached in the pool between launches */
        DRV(p_cuMemPoolSetAttribute(G.pool, CU_MEMPOOL_ATTR_RELEASE_THRESHOLD, &keep));
    }
    DRV(p_cuMemHostAlloc((void**)&G.h_counters, XMR_CTR_COUNT * sizeof(uint64_t), 0));
    G.device = device;
    G.inited = 1;
    rc = stats_reset_impl(NULL); if (rc) return rc;
    DRV(p_cuStreamSynchronize(NULL));
    const char* env = getenv("COAST_OPT_PASSES");
    if (env && !G.def_set) coast_set_opt_passes(env);
    { const char* rc_env = getenv("COAST_REPORT_COUNTERS"); static int registered;
      if (rc_env && strcmp(rc_env, "0") && !registered) { registered = 1; atexit(report_counters); } }
    return COAST_OK;
}
int coast_init(int device) { ENTER(); LEAVE(init_impl(device)); }

static int shutdown_impl(void) {
    if (!G.inited) return COAST_OK;
    ensure_ctx();
    for (int i = 0; i < 3; ++i) {
        if (G.h_in[i]) p_cuMemFree_v2(G.h_in[i]);
        if (G.h_out[i]) p_cuMemFree_v2(G.h_out[i]);
        if (G.h_aux[i]) p_cuMemFree_v2(G.h_aux[i]);
        if (G.h_stat[i]) p_cuMemFree_v2(G.h_stat[i]);
        if (G.hs[i]) p_cuStreamDestroy_v2(G.hs[i]);
        if (i == 0) { if (G.h_b) p_cuMemFree_v2(G.h_b); if (G.ev_b) p_cuEventDestroy_v2(G.ev_b); G.h_b = 0; G.h_b_cap = 0; G.ev_b = NULL; }
        G.h_in[i] = G.h_out[i] = G.h_aux[i] = G.h_stat[i] = 0;
        G.h_in_cap[i] = G.h_out_cap[i] = G.h_aux_cap[i] = G.h_stat_cap[i] = 0; G.hs[i] = NULL;
    }
    G.n_tmaps = G.tmap_next = 0;
    if (G.peer_counters) { p_cuIpcCloseMemHandle(G.peer_counters); G.peer_counters = 0; }
    p_cuMemFree_v2(G.counters);
    if (G.pool) { p_cuMemPoolDestroy(G.pool); G.pool = NULL; }
    p_cuMemFreeHost(G.h_counters);
    p_cuModuleUnload(G.mod);
    p_cuDevicePrimaryCtxRelease_v2(G.dev);
    G.inited = 0; G.n_fns = 0;
    return COAST_OK;
}
int coast_shutdown(void) { ENTER(); LEAVE(shutdown_impl()); }

/* ------------------------------------------------------------------ */
/* OPT_PASSES front end (dataflowProtection.cpp:14-47 cl::opt names)     */
/* ------------------------------------------------------------------ */
int coast_parse_opt_passes(const char* s, uint32_t* num_clones, uint32_t* flags) {
    uint32_t nc = COAST_UNPROTECTED, fl = 0; int tmr = 0, dwc = 0;
    if (!s) s = "";
    char buf[1024]; snprintf(buf, sizeof buf, "%s", s);
    for (char* tok = strtok(buf, " \t\r\n"); tok; tok = strtok(NULL, " \t\r\n")) {
        if (tok[0] == '#') break;                            /* rest of a Makefile line comment */
        if (!strcmp(tok, "-TMR")) tmr = 1;
        else if (!strcmp(tok, "-DWC")) dwc = 1;
        else if (!strcmp(tok, "-countErrors")) fl |= COAST_F_COUNT_ERRORS;
        else if (!strcmp(tok, "-countSyncs")) fl |= COAST_F_COUNT_SYNCS;
        else if (!strcmp(tok, "-noMemReplication")) fl |= COAST_F_NO_MEM_REPLICATION;
        else if (!strcmp(tok, "-storeDataSync")) fl |= COAST_F_STORE_DATA_SYNC;
        else if (!strcmp(tok, "-noStoreDataSync")) fl |= COAST_F_NO_STORE_DATA_SYNC;
        else if (!strcmp(tok, "-noLoadSync")) fl |= COAST_F_NO_LOAD_SYNC;
        else if (!strcmp(tok, "-noStoreAddrSync")) fl |= COAST_F_NO_STORE_ADDR_SYNC;
        else if (!strcmp(tok, "-i")) fl |= COAST_F_INTERLEAVE;
        else if (!strcmp(tok, "-s")) fl |= COAST_F_SEGMENT;
        else if (!strcmp(tok, "-verbose")) fl |= COAST_F_VERBOSE;
        else if (!strcmp(tok, "-reportErrors")) {
            fl |= COAST_F_REPORT_ERRORS_LEGACY;
            fprintf(stderr, "coast_rt: -reportErrors is deprecated in the reference (counts AGREEING syncs, "
                            "synchronization.cpp:1323-1350) and is not emulated; use -countErrors\n");
        }
        else fprintf(stderr, "coast_rt: OPT_PASSES token '%s' has no effect on the B200 runtime (ignored)\n", tok);
    }
    if (tmr && dwc) return fail(COAST_ERR_BAD_ARG, "-TMR and -DWC are mutually exclusive");
    if (tmr) nc = COAST_TMR; else if (dwc) nc = COAST_DWC;
    if (num_clones) *num_clones = nc;
    if (flags) *flags = fl;
    return COAST_OK;
}

static int store_votes_wanted(uint32_t fl) {
    return (fl & (COAST_F_STORE_DATA_SYNC | COAST_F_NO_MEM_REPLICATION)) && !(fl & COAST_F_NO_STORE_DATA_SYNC);
}
static int store_votes_built(uint32_t kernel) { return kernel == COAST_K_CRC16 || kernel == COAST_K_MM_U32 || kernel == COAST_K_SHA256; }

uint32_t coast_flags_honoured(uint32_t kernel, uint32_t nc, uint32_t fl) {
    uint32_t h = fl & (COAST_F_COUNT_ERRORS | COAST_F_COUNT_SYNCS | COAST_F_VERBOSE | COAST_F_MAJORITY_VOTER);
    /* layout: every kernel's native replica placement is the interleaved one (adjacent lanes of a warp; the tensor-core kernels
     * issue the replicas' MMAs back to back per k-step), so -i is what they do; replicas on separate warps (-s) exist for SHA-256 TMR only */
    h |= fl & COAST_F_INTERLEAVE;
    if (kernel == COAST_K_SHA256 && nc == 3) h |= fl & COAST_F_SEGMENT;
    if (store_votes_built(kernel))
        h |= fl & (COAST_F_NO_MEM_REPLICATION | COAST_F_STORE_DATA_SYNC | COAST_F_NO_STORE_DATA_SYNC);
    else if (!store_votes_wanted(fl))
        h |= fl & (COAST_F_NO_STORE_DATA_SYNC);              /* asking for less than what is not there is honoured trivially */
    return h;
}

int coast_set_opt_passes(const char* s) {
    uint32_t nc, fl; int rc = coast_parse_opt_passes(s, &nc, &fl);
    if (rc) return rc;
    G.def_nc = nc; G.def_flags = fl; G.def_set = 1;
    return COAST_OK;
}

/* ------------------------------------------------------------------ */
/* geometry shared with oracle/ by specification (DESIGN.md)            */
/* ------------------------------------------------------------------ */
static uint32_t sha_blocks(uint32_t len) { return (len + 8u) / 64u + 1u; }

uint32_t coast_fault_sites(uint32_t kernel, uint32_t unit_bytes, uint32_t K) {
    switch (kernel) {
    case COAST_K_CRC16:     return 2u * unit_bytes;
    case COAST_K_SHA256:    return 536u * sha_blocks(unit_bytes);
    case COAST_K_AES128:    return 176u;
    case COAST_K_MM_U32:    return K;
    case COAST_K_GEMM_TF32: return 1u;
    case COAST_K_QSORT:     return 33u * (unit_bytes / 4u);
    case COAST_K_CHSTONE_SHA: return 421u * (unit_bytes / 64u + 1u);
    case COAST_K_CHSTONE_AES: return 176u;
    default:                return 0u;
    }
}
uint32_t coast_fault_site_bits(uint32_t kernel, uint32_t unit_bytes, uint32_t K, uint32_t site) {
    (void)K;
    if (kernel == COAST_K_CRC16) return site < unit_bytes ? 16u : 8u;
    if (kernel == COAST_K_AES128 || kernel == COAST_K_CHSTONE_AES) return 8u;
    return 32u;
}
uint32_t coast_out_bytes_per_unit(uint32_t kernel) {
    static const uint32_t ob[COAST_K_COUNT_] = { 2, 32, 16, 4, 4, 0, 20, 64 };
    return kernel < COAST_K_COUNT_ ? ob[kernel] : 0;
}
uint32_t coast_votes_per_unit(uint32_t kernel) {
    static const uint32_t nv[COAST_K_COUNT_] = { 1, 32, 16, 1, 1, 0, 5, 16 };
    return kernel < COAST_K_COUNT_ ? nv[kernel] : 0;
}
uint32_t coast_out_bytes(uint32_t kernel, uint32_t unit_bytes) {
    return kernel == COAST_K_QSORT ? unit_bytes : coast_out_bytes_per_unit(kernel);
}
static uint64_t in_bytes_per_unit(const coast_launch_desc* d) {
    switch (d->kernel) {
    case COAST_K_CRC16: case COAST_K_SHA256: case COAST_K_QSORT: case COAST_K_CHSTONE_SHA: return d->unit_bytes;
    case COAST_K_AES128: return 16;
    case COAST_K_CHSTONE_AES: return 64;
    default: return 0;
    }
}
/* bytes of per-unit aux data the host call stages next to the input (AES keys) */
static uint64_t aux_bytes_per_unit(const coast_launch_desc* d) {
    if (!(d->mode & COAST_AES_KEY_PER_UNIT)) return 0;
    return d->kernel == COAST_K_AES128 ? 16 : d->kernel == COAST_K_CHSTONE_AES ? 64 : 0;
}

/* ------------------------------------------------------------------ */
/* the launch                                                           */
/* ------------------------------------------------------------------ */
static unsigned ring_smem(unsigned tile_rows, unsigned row_bytes) {
    unsigned tile = tile_rows * row_bytes;
    unsigned stride = (tile + 1023u) & ~1023u;
    return XMR_STAGES * stride + 64u;
}

static int encode_rows_map_uncached(CUtensorMap* map, const void* base, uint32_t row_bytes, uint64_t rows, uint32_t box_rows,
                                    CUtensorMapSwizzle swz) {
    cuuint64_t gdim[2] = { row_bytes / 4u, rows };
    cuuint64_t gstr[1] = { row_bytes };
    cuuint32_t box[2] = { row_bytes / 4u, box_rows };
    cuuint32_t estr[2] = { 1, 1 };
    DRV(p_cuTensorMapEncodeTiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, (void*)base, gdim, gstr, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
    return COAST_OK;
}

/* A tensor map is a pure function of (base, geometry); the host-call path re-creates the same handful every call, so the
 * last 16 are kept (round-robin replacement). */
static int encode_rows_map(CUtensorMap* map, const void* base, uint32_t row_bytes, uint64_t rows, uint32_t box_rows,
                           CUtensorMapSwizzle swz) {
    for (int i = 0; i < G.n_tmaps; ++i)
        if (G.tmaps[i].base == base && G.tmaps[i].rows == rows && G.tmaps[i].row_bytes == row_bytes &&
            G.tmaps[i].box_rows == box_rows && G.tmaps[i].swz == (int)swz) { *map = G.tmaps[i].map; return COAST_OK; }
    int rc = encode_rows_map_uncached(map, base, row_bytes, rows, box_rows, swz); if (rc) return rc;
    const int n_slots = (int)(sizeof G.tmaps / sizeof G.tmaps[0]);
    int k = G.n_tmaps < n_slots ? G.n_tmaps++ : (G.tmap_next++ % n_slots);
    G.tmaps[k].base = base; G.tmaps[k].rows = rows; G.tmaps[k].row_bytes = row_bytes; G.tmaps[k].box_rows = box_rows;
    G.tmaps[k].swz = (int)swz; G.tmaps[k].map = *map;
    return COAST_OK;
}

/* tcgen05 TF32 GEMM: A through a 2-D map (box 32 k x 128 m), B (row-major K x N, N contiguous) through a 3-D view
 * {32 n, K, N/32} (box 32 x 32 x 4) so one TMA lands the [n-chunk][k][128 B] layout the MN-major UMMA descriptor reads. */
/* tile geometry mirrors xmr::gemm::Geom<NC>: unprotected 128 x 256 tiles on 4 stages, DWC/TMR 128 x 128 on 6 stages */
static int launch_gemm_tf32(const coast_launch_desc* d, xmr_args* a, int inj, CUstream stream) {
    char name[64];
    const int wide = d->num_clones == 1 && d->N % 256u == 0;
    if (d->num_clones == 1 && !wide) snprintf(name, sizeof name, "xmr_gemm_tf32n_nc1_inj%d", inj);
    else snprintf(name, sizeof name, "xmr_gemm_tf32_nc%u_inj%d", d->num_clones, inj);
    unsigned bn = wide ? 256u : 128u, stages = wide ? 4u : 6u;
    unsigned GEMM_SMEM = stages * (16384u + 32u * bn * 4u) + 1024u + 256u;
    /* CTA-pair kernels (xmr_gemm_tf32_pair.cuh, tcgen05 cta_group::2): 256 x BN pair tiles, each CTA stages half of B.  Bit-identical
     * to the single-CTA kernels; measured at 4096^3: unprotected 0.190 vs 0.201 ms, DWC 0.320 vs 0.328 ms, TMR 0.465 vs 0.463 ms
     * (profiles/r02_gemm_pair_timings.txt).  Pairs for the unprotected and DWC kernels when the shape allows (M % 256, N % BN),
     * the single-CTA kernel for TMR. */
    unsigned b_box_chunks = 4u;
    int pair = 0;
    { const unsigned pbn = d->num_clones == 1 ? 256u : 128u;
      if (d->num_clones < 3 && d->M % 256u == 0 && d->N % pbn == 0 && G.sm_count >= 2) {
          pair = 1; bn = pbn; stages = d->num_clones == 1 ? 6u : 8u; b_box_chunks = 2u;
          GEMM_SMEM = stages * (16384u + 32u * (bn / 2u) * 4u) + 1024u + 256u;
          snprintf(name, sizeof name, "xmr_gemm_tf32p_nc%u_inj%d", d->num_clones, inj);
      } }
    CUfunction fn; int occ = 1;
    int rc = get_fn(name, GEMM_SMEM, &fn, &occ); if (rc) return rc;
    CUtensorMap ma, mb;
    {
        cuuint64_t gdim[2] = { d->K, d->M };
        cuuint64_t gstr[1] = { (cuuint64_t)d->K * 4u };
        cuuint32_t box[2] = { 32, 128 };
        cuuint32_t estr[2] = { 1, 1 };
        DRV(p_cuTensorMapEncodeTiled(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)d->d_in, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
    }
    {
        cuuint64_t gdim[3] = { 32, d->K, d->N / 32u };
        cuuint64_t gstr[2] = { (cuuint64_t)d->N * 4u, 128u };
        cuuint32_t box[3] = { 32, 32, b_box_chunks };       /* 128 columns per load; a 256-wide tile takes two (pair kernels: one half tile) */
        cuuint32_t estr[3] = { 1, 1, 1 };
        DRV(p_cuTensorMapEncodeTiled(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)d->d_aux, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
    }
    unsigned tiles = (d->M / 128u) * (d->N / bn);           /* pair kernels: CTAs = 2 x pair tiles, an even grid (cluster 2 x 1 x 1) */
    unsigned grid = tiles < (unsigned)G.sm_count ? tiles : (unsigned)G.sm_count;
    if (pair) grid &= ~1u;
    void* params[3] = { a, &ma, &mb };
    if (d->flags & COAST_F_VERBOSE) fprintf(stderr, "coast_rt: %s grid=%u smem=%u tiles=%u\n", name, grid, GEMM_SMEM, tiles);
    DRV(p_cuLaunchKernel(fn, grid, 1, 1, 384, 1, 1, GEMM_SMEM, stream, params, NULL));
    return COAST_OK;
}

/* Exact integer matmul on tcgen05 kind::i8 (xmr_mm_tc.cuh): split A and B into u8 limb planes (library scratch),
 * then ten u8 GEMMs per replica into four s32 TMEM accumulators, recombined modulo 2^32 in the epilogue. */
static int launch_mm_tc_planes(const coast_launch_desc* d, xmr_args* a, int inj, CUstream stream, int atmem, CUdeviceptr pa, CUdeviceptr pb) {
    const uint32_t nc = d->num_clones, bn = atmem ? (nc == 1 ? 64u : 32u) : (nc == 3 ? 32u : 64u);
    {
        CUfunction f; int rc = get_fn("xmr_mm_split_a", 0, &f, NULL); if (rc) return rc;
        unsigned long long rows = d->M, K = d->K; const void* A = d->d_in;
        void* params[] = { &A, &pa, &rows, &K };
        DRV(p_cuLaunchKernel(f, (unsigned)G.sm_count * 8u, 1, 1, 256, 1, 1, 0, stream, params, NULL));
        rc = get_fn("xmr_mm_split_bt", 0, &f, NULL); if (rc) return rc;
        unsigned int k32 = d->K, n32 = d->N; const void* B = d->d_aux;
        void* params2[] = { &B, &pb, &k32, &n32 };
        DRV(p_cuLaunchKernel(f, (unsigned)G.sm_count * 8u, 1, 1, 256, 1, 1, 0, stream, params2, NULL));
    }
    const unsigned smem = 2u * (65536u + 4u * bn * 128u) + 1024u + 256u;
    char name[64];
    snprintf(name, sizeof name, "xmr_mm_u32_%s_nc%u_inj%d", atmem ? "tct" : "tc", nc, inj);
    CUfunction fn; int occ = 1;
    int rc = get_fn(name, smem, &fn, &occ); if (rc) return rc;
    CUtensorMap ma, mb;
    {
        cuuint64_t gdim[3] = { d->K, d->M, 4 };
        cuuint64_t gstr[2] = { (cuuint64_t)d->K, (cuuint64_t)d->M * d->K };
        cuuint32_t box[3] = { 128, 128, 4 };
        cuuint32_t estr[3] = { 1, 1, 1 };
        DRV(p_cuTensorMapEncodeTiled(&ma, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)pa, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
    }
    {
        cuuint64_t gdim[3] = { d->K, d->N, 4 };
        cuuint64_t gstr[2] = { (cuuint64_t)d->K, (cuuint64_t)d->N * d->K };
        cuuint32_t box[3] = { 128, bn, 4 };
        cuuint32_t estr[3] = { 1, 1, 1 };
        DRV(p_cuTensorMapEncodeTiled(&mb, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)pb, gdim, gstr, box, estr,
                                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE));
    }
    unsigned tiles = (d->M / 128u) * (d->N / bn);
    unsigned grid = tiles < (unsigned)G.sm_count ? tiles : (unsigned)G.sm_count;
    void* params[3] = { a, &ma, &mb };
    if (d->flags & COAST_F_VERBOSE) fprintf(stderr, "coast_rt: %s grid=%u smem=%u tiles=%u\n", name, grid, smem, tiles);
    DRV(p_cuLaunchKernel(fn, grid, 1, 1, 256, 1, 1, smem, stream, params, NULL));
    return COAST_OK;
}
/* The limb planes (4 x u8 per element of A and of B^T) are per-launch scratch from the stream-ordered pool, like the
 * quicksort replicas: allocated on the launch's stream, released on it after the kernel, so launches on different
 * streams never share planes.  The pool keeps released memory cached, so steady state costs no driver allocation. */
static int launch_mm_tc(const coast_launch_desc* d, xmr_args* a, int inj, CUstream stream, int atmem) {
    const size_t a_bytes = (size_t)d->M * d->K * 4u, b_bytes = (size_t)d->K * d->N * 4u;   /* 4 planes of 1 byte per element */
    CUdeviceptr planes = 0;
    DRV(p_cuMemAllocFromPoolAsync(&planes, a_bytes + b_bytes, G.pool, stream));
    int rc = launch_mm_tc_planes(d, a, inj, stream, atmem, planes, planes + a_bytes);
    p_cuMemFreeAsync(planes, stream);
    return rc;
}

static int launch_impl(const coast_launch_desc* d, void* stream) {
    int rc = ensure_ctx(); if (rc) return rc;
    if (!d) return fail(COAST_ERR_BAD_ARG, "null descriptor");
    if (d->kernel >= COAST_K_COUNT_) return fail(COAST_ERR_BAD_ARG, "unknown kernel id %u", d->kernel);
    if (d->num_clones < 1 || d->num_clones > 3) return fail(COAST_ERR_BAD_ARG, "num_clones must be 1, 2 (DWC) or 3 (TMR)");
    if (d->n_units == 0) return COAST_OK;
    if (!d->d_in || !d->d_out) return fail(COAST_ERR_BAD_ARG, "null device buffer");
    const uint32_t nc = d->num_clones;
    const uint32_t upw = 32u / nc;
    const int inj = d->plan && d->plan->mode != COAST_PLAN_NONE;

    xmr_args a; memset(&a, 0, sizeof a);
    a.in = d->d_in; a.out = d->d_out; a.aux = d->d_aux;
    a.n_units = d->n_units; a.unit_base = d->unit_base;
    a.counters = (unsigned long long*)(G.peer_counters ? G.peer_counters : G.counters);
    a.status = (unsigned char*)d->d_status;
    a.unit_bytes = d->unit_bytes; a.flags = d->flags; a.mode = d->mode;
    a.M = d->M; a.N = d->N; a.K = d->K;
    memcpy(a.key, d->key, 16);
    if (inj) {
        a.plan_mode = d->plan->mode; a.seed_lo = d->plan->seed_lo; a.seed_hi = d->plan->seed_hi;
        a.threshold = d->plan->threshold; a.plan_table = (const unsigned int*)d->plan->d_table;
        if (a.plan_mode == COAST_PLAN_TABLE && !a.plan_table) return fail(COAST_ERR_BAD_ARG, "TABLE plan without d_table");
        if (a.plan_mode > COAST_PLAN_TABLE) return fail(COAST_ERR_BAD_ARG, "unknown fault plan mode %u", a.plan_mode);
    }
    a.n_sites = coast_fault_sites(d->kernel, d->unit_bytes, d->K);
    /* in-loop store votes (-storeDataSync / -noMemReplication): built for CRC16 and MM_U32, loud everywhere else */
    const int store_votes = store_votes_wanted(d->flags) && nc > 1;
    if (store_votes && !store_votes_built(d->kernel)) {
        static const char* const kname[COAST_K_COUNT_] = { "crc16", "sha256", "aes128", "mm_u32", "gemm_tf32", "qsort", "chstone_sha", "chstone_aes" };
        const char* strict = getenv("COAST_STRICT_FLAGS");
        if (strict && strcmp(strict, "0"))
            return fail(COAST_ERR_UNSUPPORTED, "-noMemReplication / -storeDataSync: the %s kernel has no in-loop store votes "
                                               "(COAST_STRICT_FLAGS is set)", kname[d->kernel]);
        if (!(G.warned_store_votes & (1u << d->kernel))) {
            G.warned_store_votes |= 1u << d->kernel;
            fprintf(stderr, "coast_rt: WARNING: -noMemReplication / -storeDataSync are NOT honoured by the %s kernel: it has no in-loop "
                            "store votes and runs the default sync set (SoR-exit votes only).  COAST_STRICT_FLAGS=1 makes this an error.\n",
                    kname[d->kernel]);
        }
    }
    if (store_votes && store_votes_built(d->kernel)) a.flags |= XMR_F_STORE_VOTES;

    char name[64];
    unsigned smem = 0; int tma = 0; int block = XMR_CTA_THREADS; int mm_tiled = 0; int qs_scratch = 0;
    unsigned tile_rows = 0, row_bytes = 0; CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_NONE;
    const int aligned16 = (((uintptr_t)d->d_in) & 15u) == 0;
    switch (d->kernel) {
    case COAST_K_SHA256:
        if (d->unit_bytes == 64 && aligned16 && d->n_units < 0x7FFFFF00ull && !store_votes) {
            tma = 1; tile_rows = XMR_WARPS * upw; row_bytes = 64; swz = CU_TENSOR_MAP_SWIZZLE_64B;
            smem = ring_smem(tile_rows, row_bytes);
            snprintf(name, sizeof name, "xmr_sha256_b64_nc%u_inj%d", nc, inj);
            /* TMR replica scheduling: -s (segmented, the reference default, interface.cpp:245-247) = replicas on
             * adjacent warps; -i (interleaved) = replicas on adjacent lanes.  Results are identical. */
            if (nc == 3 && !(d->flags & COAST_F_INTERLEAVE)) {
                block = 384; tile_rows = 128;
                smem = ((ring_smem(tile_rows, row_bytes) + 127u) & ~127u) + 2u * 4u * 2u * 8u * 32u * 4u;
                snprintf(name, sizeof name, "xmr_sha256_b64_seg_nc3_inj%d", inj);
            }
        } else {
            snprintf(name, sizeof name, "xmr_sha256_gen_nc%u_inj%d", nc, inj);
        }
        break;
    case COAST_K_CRC16:
        if (d->unit_bytes < 1 || d->unit_bytes > 255) return fail(COAST_ERR_BAD_ARG, "crc16 length is an unsigned char (1..255)");
        if (d->unit_bytes == 64 && aligned16 && d->n_units < 0x7FFFFF00ull && !store_votes) {
            /* table kernel: 1024-thread CTAs (768 unprotected), shared window = [.., 0x10000) unused | 64 KiB byte-step
             * table | tile ring at 0x20000 (CrcGeom in xmr_crc16.cuh) */
            tma = 1; block = nc == 1 ? 768 : 1024; tile_rows = (unsigned)(block / 32) * upw; row_bytes = 64;
            swz = CU_TENSOR_MAP_SWIZZLE_64B;
            smem = 0x20000u + ring_smem(tile_rows, row_bytes);
            snprintf(name, sizeof name, "xmr_crc16_b64_nc%u_inj%d", nc, inj);
        } else {
            snprintf(name, sizeof name, "xmr_crc16_gen_nc%u_inj%d", nc, inj);
        }
        break;
    case COAST_K_AES128:
        if ((d->mode & COAST_AES_KEY_PER_UNIT) && !d->d_aux) return fail(COAST_ERR_BAD_ARG, "per-unit keys need d_aux");
        if (!aligned16 || (((uintptr_t)d->d_out) & 15u)) return fail(COAST_ERR_BAD_ARG, "AES buffers must be 16-byte aligned");
        if ((d->mode & COAST_AES_KEY_PER_UNIT) && (((uintptr_t)d->d_aux) & 15u)) return fail(COAST_ERR_BAD_ARG, "AES per-unit keys must be 16-byte aligned");
        if (d->n_units >= 0x7FFFFF00ull) return fail(COAST_ERR_UNSUPPORTED, "AES: at most 2^31 - 257 blocks per launch (split the batch)");
        {
            /* one table-driven body (xmr_aes128.cuh): enc / dec with one ECB key, enck / deck with per-unit keys.  512-thread CTAs;
             * the shared window holds the ring, the two 64 KiB-aligned T-tables and, for decrypt, the 32 KiB (InvS, S) table */
            const int dec = (d->mode & COAST_AES_DECRYPT) != 0, perkey = (d->mode & COAST_AES_KEY_PER_UNIT) != 0;
            tma = 1; block = 512; tile_rows = 16u * upw * (nc == 1 ? 2u : 4u); row_bytes = 16;
            smem = dec ? 0x38000u : 0x30000u;
            static const char* const stem[4] = { "xmr_aes128_enc", "xmr_aes128_dec", "xmr_aes128_enck", "xmr_aes128_deck" };
            snprintf(name, sizeof name, "%s_nc%u_inj%d", stem[dec + 2 * perkey], nc, inj);
        }
        break;
    case COAST_K_MM_U32:
        if (!d->d_aux || !d->M || !d->N || !d->K) return fail(COAST_ERR_BAD_ARG, "MM needs A (d_in), B (d_aux) and M,N,K");
        if (d->n_units != (uint64_t)d->M * d->N) return fail(COAST_ERR_BAD_ARG, "MM: n_units must be M*N");
        snprintf(name, sizeof name, "xmr_mm_u32_nc%u_inj%d", nc, inj);
        {   /* tensor-core path (exact, u8 limbs on kind::i8) for tile-aligned problems; COAST_MM_PATH=tiled|naive overrides */
            const char* path = getenv("COAST_MM_PATH");
            const int want_tc = !path || !strcmp(path, "tc") || !strcmp(path, "tct");
            if (store_votes) break;                              /* per-k votes on `sum`: the plain kernel (one lane per replica per element) */
            if (want_tc && d->M % 128u == 0 && d->N % 64u == 0 && d->K % 128u == 0 && aligned16 &&
                !(((uintptr_t)d->d_aux) & 15u) && !(((uintptr_t)d->d_out) & 15u))
                /* measured at 4096^3: A staged in TMEM wins for TMR (1.54 vs 2.45 ms); smem operands win for 1-2 replicas */
                return launch_mm_tc(d, &a, inj, (CUstream)stream, path ? !strcmp(path, "tct") : nc == 3);
            if (path && !strcmp(path, "naive")) break;
        }
        /* register-tiled fast path: 64 x 128 x 16 tiles, NC x 128 threads (replicas on adjacent warps) */
        if (!store_votes && d->M % 64u == 0 && d->N % 128u == 0 && d->K % 16u == 0 && aligned16 && !(((uintptr_t)d->d_aux) & 15u) &&
            !(((uintptr_t)d->d_out) & 15u)) {
            mm_tiled = 1; block = (int)nc * 128; smem = 64u * 1024u;
            snprintf(name, sizeof name, "xmr_mm_u32_tiled_nc%u_inj%d", nc, inj);
        }
        break;
    case COAST_K_QSORT:
        if (d->unit_bytes < 4 || (d->unit_bytes & 3u) || d->unit_bytes > 4096u)
            return fail(COAST_ERR_BAD_ARG, "quicksort arrays are 1..1024 int32 (unit_bytes = 4*L, got %u)", d->unit_bytes);
        block = 128; qs_scratch = 1;
        snprintf(name, sizeof name, "xmr_qsort_nc%u_inj%d", nc, inj);
        break;
    case COAST_K_CHSTONE_SHA:
        if (d->unit_bytes < 64u || (d->unit_bytes & 63u) || d->unit_bytes >= (1u << 29))
            return fail(COAST_ERR_BAD_ARG, "CHStone sha streams are whole 64-byte blocks, 64 <= unit_bytes < 2^29 (got %u)", d->unit_bytes);
        if (!aligned16 || (((uintptr_t)d->d_out) & 3u)) return fail(COAST_ERR_BAD_ARG, "CHStone sha: d_in must be 16-byte and d_out 4-byte aligned");
        snprintf(name, sizeof name, "xmr_chsha_nc%u_inj%d", nc, inj);
        break;
    case COAST_K_CHSTONE_AES:
        if ((d->mode & COAST_AES_KEY_PER_UNIT) && !d->d_aux) return fail(COAST_ERR_BAD_ARG, "per-unit keys need d_aux");
        if (!aligned16 || (((uintptr_t)d->d_out) & 15u) || ((d->mode & COAST_AES_KEY_PER_UNIT) && (((uintptr_t)d->d_aux) & 15u)))
            return fail(COAST_ERR_BAD_ARG, "CHStone aes buffers must be 16-byte aligned");
        block = 512; smem = (d->mode & COAST_AES_DECRYPT) ? 0x38000u : 0x30000u;        /* same shared-memory tables as the TI kernels */
        {
            static const char* const stem[2] = { "xmr_chaes_enc", "xmr_chaes_dec" };
            snprintf(name, sizeof name, "%s_nc%u_inj%d", stem[(d->mode & COAST_AES_DECRYPT) ? 1 : 0], nc, inj);
        }
        break;
    case COAST_K_GEMM_TF32:
        if (!d->d_aux || !d->M || !d->N || !d->K) return fail(COAST_ERR_BAD_ARG, "GEMM needs A (d_in), B (d_aux) and M,N,K");
        if (d->n_units != (uint64_t)d->M * d->N) return fail(COAST_ERR_BAD_ARG, "GEMM: n_units must be M*N");
        if (d->M % 128u || d->N % 128u || d->K % 32u)
            return fail(COAST_ERR_UNSUPPORTED, "GEMM_TF32 tiles are 128x128x32: M,N must be multiples of 128 and K of 32 (got %u,%u,%u)", d->M, d->N, d->K);
        if (!aligned16 || (((uintptr_t)d->d_aux) & 15u) || (((uintptr_t)d->d_out) & 15u)) return fail(COAST_ERR_BAD_ARG, "GEMM buffers must be 16-byte aligned");
        return launch_gemm_tf32(d, &a, inj, (CUstream)stream);
    default:
        return fail(COAST_ERR_UNSUPPORTED, "kernel %u is not built into this library yet", d->kernel);
    }
    if (d->kernel == COAST_K_SHA256 && (((uintptr_t)d->d_out) & 15u)) return fail(COAST_ERR_BAD_ARG, "SHA output must be 16-byte aligned");

    CUfunction fn; int occ = 1;
    rc = get_fn_b(name, smem, block, &fn, &occ); if (rc) return rc;
    unsigned grid;
    CUtensorMap map;
    void* params[2] = { &a, &map };
    if (tma) {
        uint64_t n_tiles = (d->n_units + tile_rows - 1) / tile_rows;
        a.n_tiles = (unsigned)n_tiles;
        unsigned loads = (tile_rows + 255u) / 256u;
        while (tile_rows % loads) ++loads;                        /* mirrors TileRing::pick_loads() */
        unsigned pack = 0;                                        /* AES: the same dense bytes as 256- or 64-byte rows when the count allows */
        if (d->kernel == COAST_K_AES128) {
            pack = d->n_units % 16u == 0 ? 4u : d->n_units % 4u == 0 ? 2u : 0u;
            while (pack && (tile_rows / loads) % (1u << pack)) pack -= 2u;
            a.mode = (a.mode & ~XMR_AES_ROWPACK_MASK) | (pack << XMR_AES_ROWPACK_SHIFT);
        }
        rc = encode_rows_map(&map, d->d_in, row_bytes << pack, d->n_units >> pack, (tile_rows / loads) >> pack, swz); if (rc) return rc;
        uint64_t cap = (uint64_t)G.sm_count * (unsigned)occ;
        grid = (unsigned)(n_tiles < cap ? n_tiles : cap);
    } else if (mm_tiled) {
        grid = (d->M / 64u) * (d->N / 128u);
    } else {
        uint64_t warps = (d->n_units + upw - 1) / upw;
        uint64_t wpc = (uint64_t)block / 32u;
        uint64_t ctas = (warps + wpc - 1) / wpc;
        /* quicksort: one resident wave (persistent warps), because every warp owns a scratch slot */
        uint64_t cap = (uint64_t)G.sm_count * (unsigned)occ * (qs_scratch ? 1u : 4u);
        grid = (unsigned)(ctas < cap ? ctas : cap);
    }
    CUdeviceptr scratch = 0;
    if (qs_scratch) {
        /* private copy of every replica's array, lane-major and CONTIGUOUS per lane (a scan walks one cache line per 32
         * elements; thread-local memory would put consecutive elements of a lane 128 bytes apart) */
        size_t bytes = (size_t)grid * (size_t)(block / 32) * 32u * (size_t)d->unit_bytes;
        DRV(p_cuMemAllocFromPoolAsync(&scratch, bytes ? bytes : 4, G.pool, (CUstream)stream));
        a.aux = (const void*)scratch;
    }
    if (d->flags & COAST_F_VERBOSE)
        fprintf(stderr, "coast_rt: %s grid=%u block=%d smem=%u units=%llu\n", name, grid, block, smem,
                (unsigned long long)d->n_units);
    CUresult lr = p_cuLaunchKernel(fn, grid, 1, 1, (unsigned)block, 1, 1, smem, (CUstream)stream, params, NULL);
    if (scratch) p_cuMemFreeAsync(scratch, (CUstream)stream);           /* stream-ordered: released after the kernel */
    if (lr != CUDA_SUCCESS) return drv_fail(lr, "cuLaunchKernel");
    return COAST_OK;
}

/* ------------------------------------------------------------------ */
/* counters                                                             */
/* ------------------------------------------------------------------ */
/* Folds the device counters into *out and the reference's globals; *dwc_fired tells the guarded wrappers to call the
 * handler AFTER the single-caller guard is released (a user handler may longjmp or call back into the library). */
static int sync_impl(void* stream, coast_stats* out, int* dwc_fired) {
    int rc = ensure_ctx(); if (rc) return rc;
    if (G.peer_counters) {           /* this GPU's tallies live in the owner's block: wait for the kernels, report nothing */
        DRV(p_cuStreamSynchronize((CUstream)stream));
        if (out) { memset(out, 0, sizeof *out); out->first_fault_unit = ~0ull; }
        if (dwc_fired) *dwc_fired = 0;
        return COAST_OK;
    }
    DRV(p_cuMemcpyDtoHAsync_v2(G.h_counters, G.counters, XMR_CTR_COUNT * sizeof(uint64_t), (CUstream)stream));
    rc = stats_reset_impl(stream); if (rc) return rc;
    DRV(p_cuStreamSynchronize((CUstream)stream));
    coast_stats st;
    st.errors_corrected = G.h_counters[XMR_CTR_ERRORS];
    st.dwc_detected = G.h_counters[XMR_CTR_DWC];
    st.syncs = G.h_counters[XMR_CTR_SYNCS];
    st.injected = G.h_counters[XMR_CTR_INJECTED];
    st.first_fault_unit = G.h_counters[XMR_CTR_FIRST];
    TMR_ERROR_CNT += (uint32_t)st.errors_corrected;          /* i32 wrap, synchronization.cpp:1428-1431 */
    __SYNC_COUNT += st.syncs;
    if (out) *out = st;
    if (dwc_fired) *dwc_fired = st.dwc_detected != 0;
    return COAST_OK;
}
static int sync_guarded(void* stream, coast_stats* out, int call_handler) {
    ENTER();
    int fired = 0, rc = sync_impl(stream, out, &fired);
    leave();
    if (!rc && call_handler && fired) FAULT_DETECTED_DWC();   /* synchronization.cpp:1299-1302 */
    return rc;
}
int coast_sync(void* stream, coast_stats* out) { return sync_guarded(stream, out, 1); }
int coast_sync_noabort(void* stream, coast_stats* out) { return sync_guarded(stream, out, 0); }
int coast_launch(const coast_launch_desc* d, void* stream) { ENTER(); LEAVE(launch_impl(d, stream)); }

/* Multi-GPU counter fold in the kernels themselves (no collective): the owner exports its counter block, the other ranks
 * map it (CUDA IPC, peer access over NVLink) and every later kernel of theirs adds its tallies there with system-scope
 * atomics (Tally::flush).  The owner's coast_sync() then reads the sum over all attached GPUs; the caller orders it after
 * the other ranks' stream synchronisation (a barrier).  An attached rank's coast_sync() waits for its stream and reports zeros. */
int coast_counters_export(void* handle) {
    ENTER();
    int rc = ensure_ctx(); if (rc) LEAVE(rc);
    if (!handle) LEAVE(fail(COAST_ERR_BAD_ARG, "null handle"));
    CUipcMemHandle h;
    CUresult r = p_cuIpcGetMemHandle(&h, G.counters);
    if (r != CUDA_SUCCESS) LEAVE(drv_fail(r, "cuIpcGetMemHandle(counters)"));
    memcpy(handle, &h, sizeof h);
    LEAVE(COAST_OK);
}
int coast_counters_attach(const void* handle) {
    ENTER();
    int rc = ensure_ctx(); if (rc) LEAVE(rc);
    if (!handle) LEAVE(fail(COAST_ERR_BAD_ARG, "null handle"));
    if (G.peer_counters) LEAVE(fail(COAST_ERR_BAD_ARG, "already attached to a peer's counter block (coast_counters_detach first)"));
    CUipcMemHandle h; memcpy(&h, handle, sizeof h);
    CUdeviceptr p = 0;
    CUresult r = p_cuIpcOpenMemHandle_v2(&p, h, CU_IPC_MEM_LAZY_ENABLE_PEER_ACCESS);
    if (r != CUDA_SUCCESS) LEAVE(drv_fail(r, "cuIpcOpenMemHandle(peer counters): no peer access to the owner's GPU?"));
    G.peer_counters = p;
    LEAVE(COAST_OK);
}
int coast_counters_detach(void) {
    ENTER();
    int rc = ensure_ctx(); if (rc) LEAVE(rc);
    if (G.peer_counters) {
        CUresult r = p_cuIpcCloseMemHandle(G.peer_counters);
        G.peer_counters = 0;
        if (r != CUDA_SUCCESS) LEAVE(drv_fail(r, "cuIpcCloseMemHandle(peer counters)"));
    }
    LEAVE(COAST_OK);
}

int coast_stats_snapshot(void* stream, void* d_stats_out) {
    ENTER();
    int rc = ensure_ctx(); if (rc) LEAVE(rc);
    if (!d_stats_out) LEAVE(fail(COAST_ERR_BAD_ARG, "null d_stats_out"));
    CUresult r = p_cuMemcpyDtoDAsync_v2((CUdeviceptr)d_stats_out, G.counters, XMR_CTR_COUNT * sizeof(uint64_t), (CUstream)stream);
    LEAVE(r == CUDA_SUCCESS ? COAST_OK : drv_fail(r, "cuMemcpyDtoDAsync(counters)"));
}

/* ------------------------------------------------------------------ */
/* memory / streams / synthetic data                                    */
/* ------------------------------------------------------------------ */
int coast_malloc(void** p, size_t bytes) { int rc = ensure_ctx(); if (rc) return rc; CUdeviceptr d; DRV(p_cuMemAlloc_v2(&d, bytes ? bytes : 1)); *p = (void*)d; return COAST_OK; }
int coast_free(void* p) { int rc = ensure_ctx(); if (rc) return rc; if (p) DRV(p_cuMemFree_v2((CUdeviceptr)p)); return COAST_OK; }
int coast_memcpy_h2d(void* d, const void* h, size_t n, void* s) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuMemcpyHtoDAsync_v2((CUdeviceptr)d, h, n, (CUstream)s)); return COAST_OK; }
int coast_memcpy_d2h(void* h, const void* d, size_t n, void* s) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuMemcpyDtoHAsync_v2(h, (CUdeviceptr)d, n, (CUstream)s)); return COAST_OK; }
int coast_memset(void* d, int byte, size_t n, void* s) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuMemsetD8Async((CUdeviceptr)d, (unsigned char)byte, n, (CUstream)s)); return COAST_OK; }
int coast_host_alloc(void** h, size_t n) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuMemHostAlloc(h, n ? n : 1, 0)); return COAST_OK; }
int coast_host_free(void* h) { int rc = ensure_ctx(); if (rc) return rc; if (h) DRV(p_cuMemFreeHost(h)); return COAST_OK; }
int coast_stream_create(void** s) { int rc = ensure_ctx(); if (rc) return rc; CUstream st; DRV(p_cuStreamCreate(&st, CU_STREAM_NON_BLOCKING)); *s = st; return COAST_OK; }
int coast_stream_destroy(void* s) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuStreamDestroy_v2((CUstream)s)); return COAST_OK; }
int coast_stream_sync(void* s) { int rc = ensure_ctx(); if (rc) return rc; DRV(p_cuStreamSynchronize((CUstream)s)); return COAST_OK; }

static int fill_philox_impl(void* d_dst, uint64_t n_words, uint64_t word_base, uint32_t seed, void* stream) {
    int rc = ensure_ctx(); if (rc) return rc;
    if (!n_words) return COAST_OK;
    unsigned long long nw = n_words, wb = word_base;
    void* params[] = { &d_dst, &nw, &wb, &seed };
    uint64_t blks = (n_words + 3) / 4 + 1;
    uint64_t ctas = (blks + 255) / 256, cap = (uint64_t)G.sm_count * 16;
    return launch_small("xmr_fill_philox", (unsigned)(ctas < cap ? ctas : cap), 256, params, (CUstream)stream);
}

/* {clock64, globaltimer ns} per SM into d_out[2 * smid ..] (2 x u64 x SM count, see coast_sm_count()): two probes around a region
 * give the SM clock it really ran at.  Measurement helper of bench.py; not part of the protected path. */
int coast_clock_probe(void* d_out, void* stream) {
    ENTER();
    int rc = ensure_ctx(); if (rc) LEAVE(rc);
    if (!d_out) LEAVE(fail(COAST_ERR_BAD_ARG, "null d_out"));
    void* params[] = { &d_out };
    LEAVE(launch_small("xmr_clock_probe", 4u * (unsigned)G.sm_count, 32, params, (CUstream)stream));
}
int coast_sm_count(void) { return G.inited ? G.sm_count : 0; }

int coast_fill_philox(void* d_dst, uint64_t n_words, uint64_t word_base, uint32_t seed, void* stream) {
    ENTER(); LEAVE(fill_philox_impl(d_dst, n_words, word_base, seed, stream));
}

/* ------------------------------------------------------------------ */
/* host-buffer call: H2D -> xMR kernel -> D2H, chunked over 3 streams    */
/* ------------------------------------------------------------------ */
static int slot_reserve(CUdeviceptr* p, size_t* cap, size_t need) {
    if (*cap >= need) return COAST_OK;
    if (*p) DRV(p_cuMemFree_v2(*p));
    *p = 0; *cap = 0;
    DRV(p_cuMemAlloc_v2(p, need));
    *cap = need;
    return COAST_OK;
}

/* Device-visible alias of a HOST pointer, or 0.  Pinned host memory (cuMemHostAlloc / cudaHostAlloc / cudaHostRegister;
 * torch's pin_memory()) is mapped into the GPU's address space under UVA, so a kernel -- and the TMA unit -- can read and
 * write it over PCIe directly. */
static CUdeviceptr host_alias(const void* h, size_t bytes) {
    if (!h || !bytes) return 0;
    unsigned int mt = 0;
    if (p_cuPointerGetAttribute(&mt, CU_POINTER_ATTRIBUTE_MEMORY_TYPE, (CUdeviceptr)(uintptr_t)h) != CUDA_SUCCESS) return 0;
    if (mt != CU_MEMORYTYPE_HOST) return 0;
    CUdeviceptr d0 = 0, d1 = 0;
    if (p_cuPointerGetAttribute(&d0, CU_POINTER_ATTRIBUTE_DEVICE_POINTER, (CUdeviceptr)(uintptr_t)h) != CUDA_SUCCESS || !d0) return 0;
    /* the last byte must belong to a mapped range too (a view that runs past a registration is not ours to read) */
    if (p_cuPointerGetAttribute(&d1, CU_POINTER_ATTRIBUTE_DEVICE_POINTER, (CUdeviceptr)((uintptr_t)h + bytes - 1)) != CUDA_SUCCESS ||
        d1 != d0 + (bytes - 1)) return 0;
    return d0;
}

static int drain_host_streams(void) {
    CUresult r0 = p_cuStreamSynchronize(G.hs[0]), r1 = p_cuStreamSynchronize(G.hs[1]), r2 = p_cuStreamSynchronize(G.hs[2]);
    CUresult r = r0 != CUDA_SUCCESS ? r0 : r1 != CUDA_SUCCESS ? r1 : r2;
    return r == CUDA_SUCCESS ? COAST_OK : drv_fail(r, "cuStreamSynchronize(host-call streams)");
}

/* Chunked pipeline: H2D -> kernel -> D2H per chunk, chunks round-robin over 3 streams / 3 staging slots. */
static int run_host_staged(const coast_launch_desc* d, uint64_t ib, uint64_t ob, int per_unit_key, CUdeviceptr zin) {
    int rc;
    const uint64_t ab = aux_bytes_per_unit(d);
    const uint64_t ibs = ib ? ib : 1;                          /* divisor of the chunk schedule */
    /* each chunk is its own launch (own tensor map); the fault plan is keyed by the global unit index so
     * chunking never changes results */
    /* Chunk schedule measured on the B200 box (tools/e2e_chunk_sweep.py): 8-16 MiB chunks stream best (~12 us of driver
     * work per chunk), but a fixed size leaves the copy engines idle while the first chunk goes up and the last comes
     * down.  So chunks ramp 1,2,4,8,16,16,... MiB and shrink again towards the end (each at most half of what remains).
     * Chunks are bounded in BYTES: a unit larger than the bound (a long CHStone stream, a long SHA message) is a chunk
     * of its own, so the staging slots never exceed max(16 MiB, one unit) each. */
    uint64_t max_chunk_bytes = 16ull << 20;
    { const char* e = getenv("COAST_HOST_CHUNK_BYTES"); if (e && atoll(e) > 0) max_chunk_bytes = (uint64_t)atoll(e); }   /* tuning knob */
    const uint64_t min_chunk = ((1ull << 20) / ibs) > 1ull ? ((1ull << 20) / ibs) : 1ull;
    const uint64_t max_chunk = (max_chunk_bytes / ibs) > min_chunk ? (max_chunk_bytes / ibs) : min_chunk;
    const uint64_t chunk = max_chunk < d->n_units ? max_chunk : d->n_units;   /* slot buffers: the largest chunk this call can make */
    uint64_t ramp = min_chunk;
    uint64_t done = 0; int slot = 0;
#define STEP(call) do { CUresult r_ = (call); if (r_ != CUDA_SUCCESS) { rc = drv_fail(r_, #call); goto fail; } } while (0)
    while (done < d->n_units) {
        const uint64_t left = d->n_units - done;
        uint64_t n = ramp < max_chunk ? ramp : max_chunk;          /* ramp up */
        if (n > left / 2 && left > 2 * min_chunk) n = left / 2;    /* ramp down */
        if (n < min_chunk) n = min_chunk;
        if (n > left) n = left;
        ramp *= 2;
        rc = slot_reserve(&G.h_out[slot], &G.h_out_cap[slot], (size_t)(chunk * ob)); if (rc) goto fail;
        coast_launch_desc c = *d;
        if (zin) {                                                 /* hybrid: the kernel reads this chunk straight from mapped host memory */
            c.d_in = (void*)(zin + done * ib);
        } else {
            rc = slot_reserve(&G.h_in[slot], &G.h_in_cap[slot], (size_t)(chunk * ib) > 16 ? (size_t)(chunk * ib) : 16); if (rc) goto fail;
            if (ib) STEP(p_cuMemcpyHtoDAsync_v2(G.h_in[slot], (const uint8_t*)d->d_in + done * ib, (size_t)(n * ib), G.hs[slot]));
            c.d_in = (void*)G.h_in[slot];
        }
        c.d_out = (void*)G.h_out[slot];
        c.n_units = n; c.unit_base = d->unit_base + done;
        if (per_unit_key) {
            rc = slot_reserve(&G.h_aux[slot], &G.h_aux_cap[slot], (size_t)(chunk * ab)); if (rc) goto fail;
            STEP(p_cuMemcpyHtoDAsync_v2(G.h_aux[slot], (const uint8_t*)d->d_aux + done * ab, (size_t)(n * ab), G.hs[slot]));
            c.d_aux = (void*)G.h_aux[slot];
        }
        if (d->d_status) {                                         /* kernels index status[] chunk-locally: stage it per slot */
            rc = slot_reserve(&G.h_stat[slot], &G.h_stat_cap[slot], (size_t)chunk); if (rc) goto fail;
            c.d_status = (void*)G.h_stat[slot];
        }
        rc = launch_impl(&c, G.hs[slot]); if (rc) goto fail;
        STEP(p_cuMemcpyDtoHAsync_v2((uint8_t*)d->d_out + done * ob, G.h_out[slot], (size_t)(n * ob), G.hs[slot]));
        if (per_unit_key && d->kernel == COAST_K_AES128 && (d->mode & COAST_AES_KEY_WRITEBACK))
            STEP(p_cuMemcpyDtoHAsync_v2((uint8_t*)d->d_aux + done * 16, G.h_aux[slot], (size_t)(n * 16), G.hs[slot]));
        if (d->d_status) STEP(p_cuMemcpyDtoHAsync_v2((uint8_t*)d->d_status + done, G.h_stat[slot], (size_t)n, G.hs[slot]));
        done += n; slot = (slot + 1) % 3;
    }
#undef STEP
    return COAST_OK;
fail:
    {   /* copies of earlier chunks may still be in flight on the caller's buffers: never return before they have landed */
        char keep[sizeof G.err]; memcpy(keep, G.err, sizeof keep);
        drain_host_streams();
        memcpy(G.err, keep, sizeof keep);
    }
    return rc;
}

/* Matmul host call.  B (replicated operand) goes up once; C is produced in row blocks: block i's rows of A upload, its
 * launch and the download of its rows of C run on stream i % 3, so uploads, tensor-core work and downloads of
 * neighbouring blocks overlap (PCIe is full duplex).  The fault plan is keyed by the global element index
 * (unit_base + row * N + col), so blocking never changes results.  Small or oddly-shaped problems go in one block. */
static int run_host_matmul(const coast_launch_desc* d, coast_stats* out, int* dwc_fired) {
    int rc;
    const size_t bb = (size_t)d->K * d->N * 4;
    uint32_t blocks = 1, rows = d->M;
    { const char* hp = getenv("COAST_HOST_PATH");
      if (d->M % 128u == 0 && d->M >= 512u && !(hp && !strcmp(hp, "one-shot"))) {
          blocks = d->M / 128u < 8u ? d->M / 128u : 8u;
          rows = ((d->M / 128u + blocks - 1u) / blocks) * 128u;
          blocks = (d->M + rows - 1u) / rows;
      } }
    rc = slot_reserve(&G.h_b, &G.h_b_cap, bb); if (rc) return rc;
    if (!G.ev_b) DRV(p_cuEventCreate(&G.ev_b, CU_EVENT_DISABLE_TIMING));
    for (int i = 0; i < 3 && (uint32_t)i < blocks; ++i) {
        rc = slot_reserve(&G.h_in[i], &G.h_in_cap[i], (size_t)rows * d->K * 4); if (rc) return rc;
        rc = slot_reserve(&G.h_out[i], &G.h_out_cap[i], (size_t)rows * d->N * 4); if (rc) return rc;
    }
#define STEP(call) do { CUresult r_ = (call); if (r_ != CUDA_SUCCESS) { rc = drv_fail(r_, #call); goto fail; } } while (0)
    /* the first block of A leads on stream 0, B follows on stream 1: the first launch needs both, later blocks only their A */
    for (uint32_t i = 0; i < blocks; ++i) {
        const int slot = (int)(i % 3u);
        const uint32_t r0 = i * rows, nr = d->M - r0 < rows ? d->M - r0 : rows;
        STEP(p_cuMemcpyHtoDAsync_v2(G.h_in[slot], (const uint8_t*)d->d_in + (size_t)r0 * d->K * 4, (size_t)nr * d->K * 4, G.hs[slot]));
        if (i == 0) {
            STEP(p_cuMemcpyHtoDAsync_v2(G.h_b, d->d_aux, bb, G.hs[1]));
            STEP(p_cuEventRecord(G.ev_b, G.hs[1]));
        }
        STEP(p_cuStreamWaitEvent(G.hs[slot], G.ev_b, 0));
        coast_launch_desc c = *d;
        c.d_in = (void*)G.h_in[slot]; c.d_aux = (void*)G.h_b; c.d_out = (void*)G.h_out[slot];
        c.M = nr; c.n_units = (uint64_t)nr * d->N; c.unit_base = d->unit_base + (uint64_t)r0 * d->N;
        rc = launch_impl(&c, G.hs[slot]); if (rc) goto fail;
        STEP(p_cuMemcpyDtoHAsync_v2((uint8_t*)d->d_out + (size_t)r0 * d->N * 4, G.h_out[slot], (size_t)nr * d->N * 4, G.hs[slot]));
    }
#undef STEP
    G.last_host_path = blocks > 1 ? "row-blocks" : "one-shot";
    DRV(p_cuStreamSynchronize(G.hs[0])); DRV(p_cuStreamSynchronize(G.hs[1]));
    return sync_impl(G.hs[2], out, dwc_fired);
fail:
    { char keep[sizeof G.err]; memcpy(keep, G.err, sizeof keep); drain_host_streams(); memcpy(G.err, keep, sizeof keep); }
    return rc;
}

/* `d_in` / `d_out` / `d_aux` / `d_status` of the descriptor are HOST pointers here. */
static int run_host_impl(const coast_launch_desc* d, coast_stats* out, int* dwc_fired) {
    int rc = ensure_ctx(); if (rc) return rc;
    if (!d) return fail(COAST_ERR_BAD_ARG, "null descriptor");
    if (d->plan && d->plan->mode == COAST_PLAN_TABLE) return fail(COAST_ERR_UNSUPPORTED, "coast_run_host: TABLE plans need device pointers; use coast_launch");
    for (int i = 0; i < 3; ++i) if (!G.hs[i]) DRV(p_cuStreamCreate(&G.hs[i], CU_STREAM_NON_BLOCKING));
    const uint64_t ob = coast_out_bytes(d->kernel, d->unit_bytes);
    if (d->kernel == COAST_K_MM_U32 || d->kernel == COAST_K_GEMM_TF32) {
        if (d->d_status) return fail(COAST_ERR_UNSUPPORTED, "coast_run_host: d_status is not staged for the matmul kernels; use coast_launch");
        return run_host_matmul(d, out, dwc_fired);
    }
    const uint64_t ib = in_bytes_per_unit(d);
    /* a zero-length SHA-256 message (sha256_hash(len = 0) hashes one padded block) has nothing to stage */
    if (!ob || (!ib && d->kernel != COAST_K_SHA256)) return fail(COAST_ERR_UNSUPPORTED, "coast_run_host: kernel %u", d->kernel);
    const int per_unit_key = aux_bytes_per_unit(d) != 0;
    if (d->n_units == 0) return sync_impl(G.hs[2], out, dwc_fired);

    /* Three ways to move the bytes (COAST_HOST_PATH=staged|hybrid|zerocopy overrides the default):
     *   staged  : H2D -> kernel -> D2H per chunk over three streams (any host memory);
     *   hybrid  : pinned input + a kernel that reads each input byte once: the chunks' kernels read mapped host memory
     *             directly through the TMA ring (no upload copies, no input staging), outputs are staged and downloaded
     *             per chunk;
     *   zerocopy: ONE launch reads and WRITES mapped host memory.  Measured r02: SM stores of 16-32 bytes per lane to host
     *             memory lose to the copy engine (profiles/r02_e2e_zero_copy_experiment.md); kept for small calls. */
    const char* hp = getenv("COAST_HOST_PATH");
    const int streams_once = d->kernel == COAST_K_CRC16 || d->kernel == COAST_K_SHA256 || d->kernel == COAST_K_AES128 ||
                             d->kernel == COAST_K_CHSTONE_SHA || d->kernel == COAST_K_CHSTONE_AES;
    /* default (measured, profiles/r02_e2e_*.json): staged -- except when the output is tiny next to the input (crc16: 2 of 64 bytes,
     * CHStone sha: 20 bytes per stream), where one zero-copy launch on pinned buffers beats the chunk pipeline (1.59 vs 2.77 ms) */
    const int tiny_out = ob * 8u <= ib;
    const int want = hp ? (!strcmp(hp, "zerocopy") ? 2 : !strcmp(hp, "hybrid") ? 1 : 0) : (tiny_out ? 2 : 0);
    CUdeviceptr zin = 0;
    if (streams_once && want && ib) zin = host_alias(d->d_in, (size_t)(d->n_units * ib));
    if (want == 2 && streams_once) {
        CUdeviceptr zi = ib ? zin : (CUdeviceptr)G.counters /* never read */;
        CUdeviceptr zo = host_alias(d->d_out, (size_t)(d->n_units * ob));
        CUdeviceptr za = per_unit_key ? host_alias(d->d_aux, (size_t)(d->n_units * aux_bytes_per_unit(d))) : 0;
        CUdeviceptr zs = d->d_status ? host_alias(d->d_status, (size_t)d->n_units) : 0;
        if (zi && zo && (!per_unit_key || za) && (!d->d_status || zs)) {
            coast_launch_desc c = *d;
            c.d_in = (void*)zi; c.d_out = (void*)zo;
            if (per_unit_key) c.d_aux = (void*)za;
            if (d->d_status) c.d_status = (void*)zs;
            rc = launch_impl(&c, G.hs[2]); if (rc) return rc;
            G.last_host_path = "zerocopy";
            return sync_impl(G.hs[2], out, dwc_fired);
        }
        if (hp) return fail(COAST_ERR_BAD_ARG, "COAST_HOST_PATH=zerocopy needs pinned (mapped) host buffers");
        zin = 0;                                                   /* the default policy falls back to staged copies for pageable memory */
    }
    if (hp && want == 1 && streams_once && ib && !zin) return fail(COAST_ERR_BAD_ARG, "COAST_HOST_PATH=hybrid needs a pinned (mapped) input buffer");
    rc = run_host_staged(d, ib, ob, per_unit_key, want ? zin : 0); if (rc) return rc;
    G.last_host_path = (want && zin) ? "hybrid" : "staged";
    DRV(p_cuStreamSynchronize(G.hs[0])); DRV(p_cuStreamSynchronize(G.hs[1]));
    return sync_impl(G.hs[2], out, dwc_fired);
}
static int run_host_guarded(const coast_launch_desc* d, coast_stats* out, int call_handler) {
    ENTER();
    int fired = 0, rc = run_host_impl(d, out, &fired);
    leave();
    if (!rc && call_handler && fired) FAULT_DETECTED_DWC();   /* synchronization.cpp:1299-1302 */
    return rc;
}
const char* coast_last_host_path(void) { return G.last_host_path ? G.last_host_path : ""; }
int coast_run_host(const coast_launch_desc* d, coast_stats* out) { return run_host_guarded(d, out, 1); }
int coast_run_host_noabort(const coast_launch_desc* d, coast_stats* out) { return run_host_guarded(d, out, 0); }

/* ------------------------------------------------------------------ */
/* the four reference entry points (what the unchanged tests call)      */
/* ------------------------------------------------------------------ */
static void entry_mode(uint32_t* nc, uint32_t* fl) {
    if (!G.inited) {
        const char* dv = getenv("COAST_DEVICE");
        int rc = coast_init(dv ? atoi(dv) : 0);
        if (rc) { fprintf(stderr, "coast_rt: cannot run the protected region on a GPU: %s\n", G.err); abort(); }
    }
    if (!G.def_set) { const char* env = getenv("COAST_OPT_PASSES"); coast_set_opt_passes(env ? env : ""); }
    *nc = G.def_nc; *fl = G.def_flags;
}
static void entry_run(coast_launch_desc* d) {
    int rc = coast_run_host(d, NULL);
    if (rc) { fprintf(stderr, "coast_rt: protected launch failed: %s\n", G.err); abort(); }
}

unsigned short coast_xmr_crc16(const unsigned char* data_p, unsigned char length) {
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    unsigned short out = 0xFFFF;                               /* crc of the empty message (crc16.c:23) */
    if (!length) return out;
    d.kernel = COAST_K_CRC16; d.n_units = 1; d.unit_bytes = length; d.d_in = data_p; d.d_out = &out;
    entry_run(&d);
    return out;
}
void coast_xmr_sha256_hash(unsigned char ctx_data[], uint32_t ctx_bitlen[], uint32_t ctx_state[], unsigned char data[],
                           uint32_t len, unsigned char hash[]) {
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    unsigned char dummy = 0;
    d.kernel = COAST_K_SHA256; d.n_units = 1; d.unit_bytes = len; d.d_in = len ? data : &dummy; d.d_out = hash;
    entry_run(&d);
    /* The caller-visible scratch the reference leaves behind (sha256_common_tmr.c:101-180): replicas keep it in registers,
     * so it is rebuilt here from the voted digest and the message -- marshalling, not computation.
     *   ctx_state : the final chaining value = the digest words, big-endian (:169-178)
     *   ctx_bitlen: {low, high} of 8*len (DBL_INT_ADD, :124,155)
     *   ctx_data  : the last block fed to sha256_transform (:132-163) */
    if (ctx_state)
        for (int i = 0; i < 8; ++i)
            ctx_state[i] = ((uint32_t)hash[4 * i] << 24) | ((uint32_t)hash[4 * i + 1] << 16) | ((uint32_t)hash[4 * i + 2] << 8) | hash[4 * i + 3];
    const uint32_t lo = len << 3, hi = len >> 29;
    if (ctx_bitlen) { ctx_bitlen[0] = lo; ctx_bitlen[1] = hi; }
    if (ctx_data) {
        const uint32_t rem = len & 63u;
        if (rem < 56u) {
            memcpy(ctx_data, data + (len - rem), rem);
            ctx_data[rem] = 0x80; memset(ctx_data + rem + 1, 0, 55u - rem);
        } else {
            memset(ctx_data, 0, 56);                               /* the extra block: sha_memset(ctx_data, 0, 56) :142-150 */
        }
        ctx_data[63] = (unsigned char)lo; ctx_data[62] = (unsigned char)(lo >> 8); ctx_data[61] = (unsigned char)(lo >> 16); ctx_data[60] = (unsigned char)(lo >> 24);
        ctx_data[59] = (unsigned char)hi; ctx_data[58] = (unsigned char)(hi >> 8); ctx_data[57] = (unsigned char)(hi >> 16); ctx_data[56] = (unsigned char)(hi >> 24);
    }
}
void coast_xmr_aes_enc_dec(unsigned char* state, unsigned char* key, unsigned char dir) {
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    /* per-unit-key mode with write-back so key[] is mutated exactly as TI_aes_128.c:107-231 does */
    d.kernel = COAST_K_AES128; d.n_units = 1; d.d_in = state; d.d_out = state; d.d_aux = key;
    d.mode = (dir ? COAST_AES_DECRYPT : 0) | COAST_AES_KEY_PER_UNIT | COAST_AES_KEY_WRITEBACK;
    entry_run(&d);
}
void coast_xmr_chstone_sha_stream(const unsigned char* indata, const int* in_i, int vsize, int block_size, uint32_t* digest) {
    /* sha_stream (sha.c:182-193) feeds chunk j = indata[j][0 .. in_i[j]) to sha_update; with whole-block chunks that is the
     * hash of the concatenation, which is what one unit of the kernel computes */
    size_t total = 0;
    for (int j = 0; j < vsize; ++j) {
        if (in_i[j] < 0 || in_i[j] > block_size || (in_i[j] & 63)) {
            fprintf(stderr, "coast_rt: sha_stream chunk %d has %d bytes; only whole 64-byte blocks are supported\n", j, in_i[j]);
            abort();
        }
        total += (size_t)in_i[j];
    }
    unsigned char* cat = (unsigned char*)malloc(total ? total : 1);
    if (!cat) abort();
    size_t off = 0;
    for (int j = 0; j < vsize; ++j) { memcpy(cat + off, indata + (size_t)j * (size_t)block_size, (size_t)in_i[j]); off += (size_t)in_i[j]; }
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    d.kernel = COAST_K_CHSTONE_SHA; d.n_units = 1; d.unit_bytes = (uint32_t)total; d.d_in = cat; d.d_out = digest;
    entry_run(&d);
    free(cat);
}
void coast_xmr_chstone_aes(int* statemt, const int* key, int type, int dir) {
    if (type != 128128) {
        fprintf(stderr, "coast_rt: chstone/aes type %d: only 128128 (the benchmark's, aes.c:126-127) has a protected kernel\n", type);
        abort();
    }
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    /* 16-byte aligned bounce buffers: the program's statemt[] / key[] are plain int arrays */
    int st[16] __attribute__((aligned(16))), k[16] __attribute__((aligned(16)));
    memcpy(st, statemt, sizeof st); memcpy(k, key, sizeof k);
    d.kernel = COAST_K_CHSTONE_AES; d.n_units = 1; d.d_in = st; d.d_out = st; d.d_aux = k;
    d.mode = (dir ? COAST_AES_DECRYPT : 0) | COAST_AES_KEY_PER_UNIT;
    entry_run(&d);
    memcpy(statemt, st, sizeof st);
}
void coast_xmr_matrix_multiply_u32(const uint32_t* f, const uint32_t* s, uint32_t* r, int side) {
    coast_launch_desc d; memset(&d, 0, sizeof d);
    entry_mode(&d.num_clones, &d.flags);
    d.kernel = COAST_K_MM_U32; d.M = d.N = d.K = (uint32_t)side; d.n_units = (uint64_t)side * side;
    d.d_in = f; d.d_aux = s; d.d_out = r;
    entry_run(&d);
}
