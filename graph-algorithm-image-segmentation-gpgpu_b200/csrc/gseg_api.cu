// gseg_api.cu -- host side of libgseg.so: context, round scheduling, the C-ABI of include/gseg.h.
//
// There is no CPU path in this file: every compute entry point launches the CUDA kernels of
// gseg_kernels.cuh and fails with GSEG_E_CUDA when no device is usable.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvjpeg.h> // types and prototypes only: the library is loaded with dlopen on first use
#include <limits.h>
#include <stddef.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/gseg.h"
#include "gseg_kernels.cuh"
#include "gseg_regions.cuh"
#include "gseg_sort.cuh"
#include "gseg_dedup.cuh"
#include "gseg_jpeg.hpp"
#include "gseg_jpeg.cuh"

#define GSEG_MAXMARK 1024
#define GRID_CAP (148 * 8)

// Host-initialised head of GsegCtl (layout-compatible prefix).
struct GsegHead {
    GsegRunParams p;
    RoundState st;
    u32 Vnext, error, ticketC, ticketE, doneE, Eacc[GSEG_MAXR + 1];
    u32 map_skip[GSEG_MAXR + 1], resume_phase;
    u32 stDedupIn[GSEG_MAXR + 1], stDedupOut[GSEG_MAXR + 1];
};
static_assert(offsetof(GsegCtl, Eacc) == offsetof(GsegHead, Eacc), "GsegHead must mirror the head of GsegCtl");
static_assert(offsetof(GsegCtl, resume_phase) == offsetof(GsegHead, resume_phase), "GsegHead must mirror the head of GsegCtl");
static_assert(offsetof(GsegCtl, stDedupOut) == offsetof(GsegHead, stDedupOut), "GsegHead must mirror the head of GsegCtl");
#define GSEG_EPOCHS_PER_RUN (2u * GSEG_MAXR + 8u + 32u) /* look-back tags a run may use: 2 per round, 8 spare, 32 de-duplications */

// Staging the next page in shared memory pays while a warp has few pages: the pool's images (7 pages per warp at
// 1080p, ~55 for 4K 8-connected) ran 3-4 % faster end to end; one 2^30-pixel image alone (~1 800 pages per warp)
// ran 0.9 % slower, so beyond this many pages per warp the rows are loaded straight into registers.
#define R0_STAGE_MAX_PPW 128

// Region statistics: partitions with at most this many components accumulate in a block-private shared-memory table
// (40 bytes per component: 40 KB at 1024, which leaves 5 blocks of 256 threads per SM); above it every warp's combined
// runs go straight to 64-bit global atomics.  At 1024 components a block still sees only the few dozen regions its rows
// cross, so the flush (one pass over the table, atomics for the non-empty records) stays small against its pixels.
#define REGIONS_SMEM_MAX 1024

static const size_t TAIL_SMEM = (2 * (size_t)GSEG_TAIL_STAGE + 2 * (NTT / 32)) * sizeof(u32); // k_tail: staged map + minima, survivor-count exchange (phase_E)

struct gseg_ctx {
    int device, max_w, max_h;
    size_t Vmax;
    int Dmax; // directions the context was sized for (2: 4-connected only, 4: 8-connected too)
    cudaStream_t stream, own_stream;
    uint8_t *d_rgb;
    float *d_tmp, *d_planes, *d_G, *d_wgrid;
    u32 *d_wsel, *d_succ, *d_rank;
    u64 *d_best[2];
    uint2 *d_attr[2];
    long long *d_csum[2];
    float4 *d_cmean[2];
    uint2 *d_eab[2];
    u32 *d_ew[2], *d_pcnt[2], *d_poff[2], *d_pscan;
    u32 *d_arena;
    size_t arena_cap;
    u64 *d_statusC, *d_statusE;
    size_t ntilesC, ntilesE;
    int *d_labels[2];
    GsegCtl *d_ctl, *h_ctl;
    GsegHead *h_head; // pinned image of the host-initialised head of the control block
    int num_sms, occ_mult;
    u32 filter_shift;
    u32 r0_stage_ppw;     // round-0 edge kernel: most pages per warp for the staged body (GSEG_R0_STAGE_PPW)
    u32 rg_smem_max;      // region statistics: most components of the shared-memory tier (GSEG_REGIONS_SMEM_MAX)
    u32 rg_smem_fit;      // ... and most the device's shared memory per block holds
    u32 rg_n;             // components of the last region table (profile byte model)
    u64 *d_rtab;          // region table staging for host output when d_best[0] is too small (GSEG_CAP_REGIONS)
    int tail_cluster;     // CTAs in the tail kernel's cluster (16 non-portable, else 8)
    bool tail_cluster_env; // GSEG_TAIL_CLUSTER was given: a pool leaves the size alone
    u32 tail_E, tail_V, tail_P; // hand-over thresholds of the tail kernel
    u32 run_tail_E, run_tail_V; // thresholds the last run used
    int nbig_hint;        // grid-wide rounds to enqueue before the tail (-1: estimate; adapts to the last run)
    int hint_w, hint_h, hint_variant, hint_conn;
    SortScratch sort;
    // duplicate elimination between rounds (gseg_dedup.cuh): descriptor in device memory, arrays of dd_cap edges
    DedupDev *d_dd;
    u64 *d_winner;
    size_t dd_cap;
    u32 dd_min_edges, dd_min_ratio, dd_V;
    bool dd_on;
    bool dd_skip; // the last image of this shape never triggered the elimination: do not enqueue its (self-skipping) launches again
    // export of the final component graph (tiled schedule): cached dense / de-duplicated edge list; shares the
    // arrays below with the duplicate elimination
    u64 *d_xkeys;
    u32 *d_xvals, *d_xkeep, *d_xw, *x_w;
    uint2 *d_xab, *x_ab;
    size_t x_cap, x_count;
    bool x_valid, x_dedup;
    // run state
    gseg_params params;
    int w, h, D;
    bool valid, pending;
    bool graph_mode;              // the last run was gseg_segment_graph (rounds numbered from 1, no pixel map)
    bool strip_labels;            // d_labels[0] holds the dense labels of the strip gseg_strip_record described
    int strip_w, strip_h, halo_top;
    u32 strip_nV;
    long long compactions;        // arena compactions since creation (FELZ)
    bool rgb_staged;              // the last run read its input from d_rgb (host input or JPEG)
    nvjpegHandle_t jpg_handle; nvjpegJpegState_t jpg_state; // nvJPEG objects, created on first gseg_segment_jpeg
    // in-house JPEG decoder (gseg_jpeg.cuh): staged file bytes, descriptor + interval starts, coefficients, sample planes
    uint8_t *d_jfile, *d_jsamples, *h_jdesc;
    JpegDev *d_jdev;
    int16_t *d_jcoef;
    size_t jfile_cap, jsamples_cap, jdev_cap, jcoef_cap, hjdesc_cap;
    uint8_t *d_jsub;              // sub-sequence states of the marker-less decode (k_jpeg_sync): entry, exit, counts, flags
    size_t jsub_cap;
    uint32_t jsub_bytes;          // bytes per sub-sequence (GSEG_JPEG_SUB, default 128)
    bool jsync_grid;              // marker-less decode as a grid of small blocks with a software barrier (GSEG_JPEG_SYNC=grid) instead of one cluster
    uint32_t *d_jerr;             // [2] JPG_ERR_* bits of the last two decodes (ping-pong)
    cudaEvent_t ev_jdesc;         // the last descriptor copy out of h_jdesc
    cudaEvent_t ev_jdone;         // end of the last decode (its buffers are free again)
    int jerr_next;                // which of the two error words the next decode takes
    int jflag_slot;               // error word the next segmentation hands to its control block (-1: none)
    int jpeg_backend, jpeg_used;  // GSEG_JPEG_*: what the caller asked for / what the last JPEG run used
    JpegPlan *jplan;
    u32 epoch_next;
    char err[256];
    // per-kernel profiling (host-driven schedule only) and launch accounting
    bool profiling;
    int n_marks;
    cudaEvent_t ev[GSEG_MAXMARK + 1];
    const char *mark_name[GSEG_MAXMARK];
    int mark_round[GSEG_MAXMARK];
    long long launches, graph_nodes;
};

static int fail(gseg_ctx *c, int code, const char *what, cudaError_t e) {
    if (c) snprintf(c->err, sizeof(c->err), "%s: %s", what, e == cudaSuccess ? "" : cudaGetErrorString(e));
    return code;
}
#define CK(call)                                                              \
    do {                                                                      \
        cudaError_t e__ = (call);                                             \
        if (e__ != cudaSuccess) return fail(ctx, GSEG_E_CUDA, #call, e__);    \
    } while (0)

extern "C" int gseg_version(void) { return GSEG_VERSION; }

extern "C" const char *gseg_strerror(int s) {
    switch (s) {
    case GSEG_OK: return "ok";
    case GSEG_E_ARG: return "bad argument";
    case GSEG_E_CUDA: return "CUDA error or no CUDA device (there is no CPU fallback)";
    case GSEG_E_SIZE: return "image larger than the context capacity";
    case GSEG_E_ARENA: return "supervertex-map arena exhausted";
    case GSEG_E_INTERNAL: return "device-side watchdog tripped";
    case GSEG_E_STATE: return "no completed segmentation in this context";
    case GSEG_E_LEVEL: return "hierarchy level out of range";
    case GSEG_E_UNSUPPORTED: return "optional dependency missing at run time";
    case GSEG_E_RANGE: return "label type too narrow for the component count, or output buffer too small";
    default: return "unknown status";
    }
}
extern "C" const char *gseg_last_error(const gseg_ctx *ctx) { return ctx ? ctx->err : "null context"; }

static inline int grid_for(size_t n, int per_block, int cap = GRID_CAP) {
    size_t g = (n + per_block - 1) / per_block;
    if (g < 1) g = 1;
    if (g > (size_t)cap) g = cap;
    return (int)g;
}

template <typename T>
static cudaError_t dalloc(T **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(T)); }

// Largest cluster size <= want that the device can co-schedule for the tail kernel.
static int fit_tail_cluster(int want) {
    if (want < 1) want = 1;
    if (want > 16) want = 16;
    for (; want > 1; --want) {
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute at[1];
        cfg.gridDim = dim3(want); cfg.blockDim = dim3(NTT); cfg.dynamicSmemBytes = TAIL_SMEM;
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = want; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int ncl = 0;
        if (cudaOccupancyMaxActiveClusters(&ncl, k_tail<true>, &cfg) == cudaSuccess && ncl >= 1) break;
        cudaGetLastError();
    }
    return want;
}

// The de-duplication's descriptor: pointers into the context's arrays (re-sent when a sort grew the scratch).
static cudaError_t upload_dd(gseg_ctx *ctx) {
    DedupDev dd;
    memset(&dd, 0, sizeof(dd));
    dd.sort.keys[0] = ctx->d_xkeys; dd.sort.keys[1] = ctx->sort.keys_alt;
    dd.sort.vals[0] = ctx->d_xvals; dd.sort.vals[1] = ctx->sort.vals_alt;
    dd.sort.hist = ctx->sort.hist; dd.sort.status = ctx->sort.status; dd.sort.tickets = ctx->sort.tickets;
    dd.xab = ctx->d_xab; dd.xw = ctx->d_xw; dd.winner = ctx->d_winner; dd.keep = ctx->d_xkeep;
    const size_t cap = ctx->dd_cap < ctx->sort.cap_n ? ctx->dd_cap : ctx->sort.cap_n;
    dd.cap = (u32)cap; dd.min_edges = ctx->dd_min_edges; dd.min_ratio = ctx->dd_min_ratio; dd.disabled = ctx->dd_on ? 0u : 1u;
    return cudaMemcpy(ctx->d_dd, &dd, sizeof(dd), cudaMemcpyHostToDevice);
}

extern "C" int gseg_create(gseg_ctx **out, int device, int max_w, int max_h) {
    return gseg_create_ex(out, device, max_w, max_h, 8);
}

extern "C" int gseg_create_ex(gseg_ctx **out, int device, int max_w, int max_h, int max_connectivity) {
    if (!out || max_w < 1 || max_h < 1 || (max_connectivity != 4 && max_connectivity != 8)) return GSEG_E_ARG;
    *out = nullptr;
    const size_t V = (size_t)max_w * (size_t)max_h;
    const size_t Dmax = max_connectivity == 8 ? 4 : 2;
    if ((V / GSEG_PAGE + 2) * GSEG_PAGE * Dmax >= 0xFFFFFFFFull) return GSEG_E_SIZE; // 32-bit edge indices and list slots
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return GSEG_E_CUDA;
    gseg_ctx *ctx = (gseg_ctx *)calloc(1, sizeof(gseg_ctx));
    if (!ctx) return GSEG_E_ARG;
    ctx->device = device; ctx->max_w = max_w; ctx->max_h = max_h; ctx->Vmax = V; ctx->Dmax = (int)Dmax;
    ctx->epoch_next = 1; ctx->jflag_slot = -1;
    ctx->jsub_bytes = 128u;
    if (const char *ev = getenv("GSEG_JPEG_SYNC")) ctx->jsync_grid = !strcmp(ev, "grid");
    if (const char *ev = getenv("GSEG_JPEG_SUB")) { const int v = atoi(ev); if (v >= 8 && v <= 65536) ctx->jsub_bytes = (uint32_t)v; }
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    ctx->stream = ctx->own_stream;
    const size_t Vp = V + 64; // slack for vector tails
    const size_t Eslots = Dmax * ((V + GSEG_PAGE - 1) / GSEG_PAGE + 1) * GSEG_PAGE;
    const size_t Pslots = Dmax * (V / GSEG_PAGE + 1) + 8;
    if (e == cudaSuccess) e = dalloc(&ctx->d_rgb, 3 * Vp);
    if (e == cudaSuccess) e = dalloc(&ctx->d_planes, 3 * Vp);
    if (e == cudaSuccess) e = dalloc(&ctx->d_wgrid, Dmax * Vp);
    if (e == cudaSuccess) e = dalloc(&ctx->d_wsel, Vp);
    if (e == cudaSuccess) e = dalloc(&ctx->d_succ, Vp);
    if (e == cudaSuccess) e = dalloc(&ctx->d_rank, Vp);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = dalloc(&ctx->d_best[i], Vp);
        if (e == cudaSuccess) e = dalloc(&ctx->d_attr[i], Vp);
        // paged edge list: up to 4 directions x ceil(V / page) pages of GSEG_PAGE slots
        if (e == cudaSuccess) e = dalloc(&ctx->d_eab[i], Eslots);
        if (e == cudaSuccess) e = dalloc(&ctx->d_ew[i], Eslots);
        if (e == cudaSuccess) e = dalloc(&ctx->d_pcnt[i], Pslots);
        if (e == cudaSuccess) e = dalloc(&ctx->d_poff[i], Pslots);
    }
    if (e == cudaSuccess) e = dalloc(&ctx->d_pscan, Pslots);
    // one old->new map per round: V + V1 + V2 + ... ; 6V covers every input up to 2^26 pixels, above that the
    // arena is 2.5V (a run that needs more ends with GSEG_E_ARENA) so that a 2^30-pixel context fits in HBM
    ctx->arena_cap = V <= ((size_t)1 << 26) ? 6 * V + 1024 : V * 5 / 2 + 1024;
    if (const char *ev = getenv("GSEG_ARENA_FACTOR")) { // test knob: arena entries per pixel (exercises the compaction)
        const double f = atof(ev);
        if (f >= 1.0 && f <= 16.0) ctx->arena_cap = (size_t)(f * (double)V) + 64;
    }
    if (ctx->arena_cap > 0xFFFFFFF0ull) ctx->arena_cap = 0xFFFFFFF0ull;
    if (e == cudaSuccess) e = dalloc(&ctx->d_arena, ctx->arena_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_labels[0], Vp); // staging of label images that go to host memory
    // look-back status words: one per tile of the largest tiling that uses each array
    ctx->ntilesC = V / (32 * CPT) + 2;
    const size_t img_tiles = (size_t)((max_w + TW - 1) / TW) * (size_t)((max_h + GH - 1) / GH); // round-0 graph tiles
    if (ctx->ntilesC < img_tiles) ctx->ntilesC = img_tiles;
    ctx->ntilesE = Pslots; // pages of the edge list
    if (e == cudaSuccess) e = dalloc(&ctx->d_statusC, ctx->ntilesC);
    if (e == cudaSuccess) e = dalloc(&ctx->d_statusE, ctx->ntilesE);
    if (e == cudaSuccess) e = cudaMemset(ctx->d_statusC, 0, ctx->ntilesC * sizeof(u64));
    if (e == cudaSuccess) e = cudaMemset(ctx->d_statusE, 0, ctx->ntilesE * sizeof(u64));
    if (e == cudaSuccess) e = dalloc(&ctx->d_ctl, 1);
    if (e == cudaSuccess) e = cudaMemset(ctx->d_ctl, 0, sizeof(GsegCtl));
    // duplicate elimination / graph export: arrays for up to dd_cap edges (it runs once V <= 65536, when the list has
    // shrunk far below the grid's edge count), sort scratch included -- nothing of this allocates later
    ctx->dd_cap = V < ((size_t)1 << 24) ? V : ((size_t)1 << 24);
    if (ctx->dd_cap < 4096) ctx->dd_cap = 4096;
    // Thresholds from measurements on B200 (DESIGN.md section 2 item 7): the sort pays once the graph is down to <= 4096
    // components (two 12-bit ids: three 8-bit passes) while the list still holds >= 2^19 edges (4K 8-connected
    // hierarchies, large images); below that the remaining rounds cost less than the sort and it does not run.
    ctx->dd_on = true; ctx->dd_min_edges = 1u << 19; ctx->dd_min_ratio = 8u; ctx->dd_V = 4096u;
    if (const char *ev = getenv("GSEG_DEDUP_V")) ctx->dd_V = (u32)strtoul(ev, nullptr, 10);
    if (const char *ev = getenv("GSEG_DEDUP")) ctx->dd_on = atoi(ev) != 0;
    if (const char *ev = getenv("GSEG_DEDUP_MIN")) ctx->dd_min_edges = (u32)strtoul(ev, nullptr, 10);
    if (const char *ev = getenv("GSEG_DEDUP_RATIO")) ctx->dd_min_ratio = (u32)strtoul(ev, nullptr, 10);
    if (e == cudaSuccess) e = dalloc(&ctx->d_xkeys, ctx->dd_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_xvals, ctx->dd_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_xkeep, ctx->dd_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_xab, ctx->dd_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_xw, ctx->dd_cap);
    if (e == cudaSuccess) e = dalloc(&ctx->d_winner, ctx->dd_cap);
    if (e == cudaSuccess) { ctx->x_cap = ctx->dd_cap; e = sort_scratch_reserve(&ctx->sort, ctx->dd_cap); }
    if (e == cudaSuccess) e = dalloc(&ctx->d_dd, 1);
    if (e == cudaSuccess) e = upload_dd(ctx);
    if (e == cudaSuccess) e = cudaMallocHost((void **)&ctx->h_ctl, sizeof(GsegCtl));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&ctx->h_head, sizeof(GsegHead));
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) {
        // tail kernel: one thread-block cluster, 16 CTAs when the device can co-schedule that many
        cudaFuncSetAttribute(k_tail<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaFuncSetAttribute(k_tail<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        int want = 16;
        cudaFuncSetAttribute(k_tail<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TAIL_SMEM);
        cudaFuncSetAttribute(k_tail<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TAIL_SMEM);
        if (const char *ev = getenv("GSEG_TAIL_CLUSTER")) want = atoi(ev);
        ctx->tail_cluster = fit_tail_cluster(want);
        ctx->tail_cluster_env = getenv("GSEG_TAIL_CLUSTER") != nullptr;
        ctx->tail_E = 256u * 1024u; ctx->tail_V = 64u * 1024u; ctx->tail_P = 4096u;
        if (const char *ev = getenv("GSEG_TAIL_P")) ctx->tail_P = (u32)strtoul(ev, nullptr, 10);
        if (const char *ev = getenv("GSEG_TAIL_E")) ctx->tail_E = (u32)strtoul(ev, nullptr, 10);
        if (const char *ev = getenv("GSEG_TAIL_V")) ctx->tail_V = (u32)strtoul(ev, nullptr, 10);
        ctx->nbig_hint = -1;
        ctx->occ_mult = 4;
        if (const char *ev = getenv("GSEG_OCC_MULT")) ctx->occ_mult = atoi(ev) > 0 ? atoi(ev) : 4;
        ctx->filter_shift = 6;
        if (const char *ev = getenv("GSEG_FILTER_SHIFT")) ctx->filter_shift = (u32)atoi(ev);
        ctx->r0_stage_ppw = R0_STAGE_MAX_PPW; // test knob: 0 = always the register body, huge = always the staged one
        if (const char *ev = getenv("GSEG_R0_STAGE_PPW")) ctx->r0_stage_ppw = (u32)strtoul(ev, nullptr, 10);
        ctx->rg_smem_max = REGIONS_SMEM_MAX; // test knob: 0 = always the global-atomic tier, huge = shared memory whenever it fits
        if (const char *ev = getenv("GSEG_REGIONS_SMEM_MAX")) ctx->rg_smem_max = (u32)strtoul(ev, nullptr, 10);
        int optin = 0;
        e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_regions<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
        ctx->rg_smem_fit = (u32)optin / (RG_FIELDS * sizeof(u32));
    }
    if (e != cudaSuccess) {
        fprintf(stderr, "gseg_create: %s\n", cudaGetErrorString(e));
        gseg_destroy(ctx);
        return GSEG_E_CUDA;
    }
    memset(ctx->h_ctl, 0, sizeof(GsegCtl));
    *out = ctx;
    return GSEG_OK;
}


// ---- nvJPEG (optional, dlopen) ------------------------------------------------------------------------
// JPEG input decoded on the GPU into the staged RGB buffer (SURVEY.md s8f N2).  Library code, outside
// the hot path; libgseg.so has no link-time dependency on it.
struct NvJpegApi {
    void *lib;
    decltype(&nvjpegCreateSimple) create;
    decltype(&nvjpegDestroy) destroy;
    decltype(&nvjpegJpegStateCreate) state_create;
    decltype(&nvjpegJpegStateDestroy) state_destroy;
    decltype(&nvjpegGetImageInfo) info;
    decltype(&nvjpegDecode) decode;
    bool ok;
};
static NvJpegApi *nvjpeg_api() {
    static NvJpegApi api = [] {
        NvJpegApi a = {};
        const char *names[] = {"libnvjpeg.so.12", "libnvjpeg.so"};
        for (const char *n : names)
            if ((a.lib = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
        if (!a.lib) return a;
        a.create = (decltype(a.create))dlsym(a.lib, "nvjpegCreateSimple");
        a.destroy = (decltype(a.destroy))dlsym(a.lib, "nvjpegDestroy");
        a.state_create = (decltype(a.state_create))dlsym(a.lib, "nvjpegJpegStateCreate");
        a.state_destroy = (decltype(a.state_destroy))dlsym(a.lib, "nvjpegJpegStateDestroy");
        a.info = (decltype(a.info))dlsym(a.lib, "nvjpegGetImageInfo");
        a.decode = (decltype(a.decode))dlsym(a.lib, "nvjpegDecode");
        a.ok = a.create && a.destroy && a.state_create && a.state_destroy && a.info && a.decode;
        return a;
    }();
    return api.ok ? &api : nullptr;
}
static void jpeg_release(gseg_ctx *ctx) {
    if (!ctx->jpg_state && !ctx->jpg_handle) return; // JPEG never used: do not even load the library
    NvJpegApi *a = nvjpeg_api();
    if (!a) return;
    if (ctx->jpg_state) a->state_destroy(ctx->jpg_state);
    if (ctx->jpg_handle) a->destroy(ctx->jpg_handle);
    ctx->jpg_state = nullptr; ctx->jpg_handle = nullptr;
}
static int jpeg_size(NvJpegApi *a, nvjpegHandle_t hnd, const void *jpeg, size_t nbytes, int *w, int *h) {
    int ncomp = 0, ws[NVJPEG_MAX_COMPONENT] = {0}, hs[NVJPEG_MAX_COMPONENT] = {0};
    nvjpegChromaSubsampling_t sub;
    if (a->info(hnd, (const unsigned char *)jpeg, nbytes, &ncomp, &sub, ws, hs) != NVJPEG_STATUS_SUCCESS || ws[0] < 1 || hs[0] < 1)
        return GSEG_E_ARG;
    *w = ws[0]; *h = hs[0];
    return GSEG_OK;
}

extern "C" int gseg_jpeg_info(const void *jpeg, size_t nbytes, int *w, int *h) {
    if (!jpeg || !nbytes || !w || !h) return GSEG_E_ARG;
    return jpeg_peek_size((const uint8_t *)jpeg, nbytes, w, h) == JPG_OK ? GSEG_OK : GSEG_E_ARG; // header parse on the host
}

#define GSEG_JPEG_SYNC_MIN_RI 8 // restart intervals longer than this many MCUs are not decoded one thread per interval but as
                                // self-synchronising sub-sequences (1080p 4:2:0: 0.8 ms at 8 MCUs per thread, 1.2 ms for the other way)
// ---- in-house decoder (gseg_jpeg.cuh) -------------------------------------------------------------------
// (Re)allocates one of the decoder's device buffers; growing waits for the last decode first (rare: the buffers are
// sized for the context's capacity by the first JPEG or by gseg_reserve(GSEG_CAP_JPEG)).
template <typename T>
static int jpeg_grow(gseg_ctx *ctx, T **p, size_t *cap, size_t need, size_t want) {
    if (*p && *cap >= need) return GSEG_OK;
    if (want < need) want = need;
    if (*p) {
        if (ctx->ev_jdone) CK(cudaEventSynchronize(ctx->ev_jdone));
        cudaFree(*p); *p = nullptr; *cap = 0;
    }
    CK(cudaMalloc((void **)p, want * sizeof(T)));
    *cap = want;
    return GSEG_OK;
}
static int jpeg_reserve_own(gseg_ctx *ctx, size_t file_bytes, size_t nint, size_t nblocks) {
    // default sizes: any 4:4:4 image of the context's capacity with one MCU per restart interval
    const size_t V = ctx->Vmax, side = (size_t)(ctx->max_w + ctx->max_h);
    const size_t blocks_max = 3 * (V / 64 + side / 2 + 64);
    int rc = jpeg_grow(ctx, &ctx->d_jfile, &ctx->jfile_cap, file_bytes + 64, V + 4096);
    if (!rc && (!ctx->d_jcoef || ctx->jcoef_cap < nblocks * 64)) {
        rc = jpeg_grow(ctx, &ctx->d_jcoef, &ctx->jcoef_cap, nblocks * 64, blocks_max * 64);
        // all zero between images: the Huffman threads write non-zero coefficients only, k_jpeg_idct clears what it read
        if (!rc) {
            CK(cudaMemsetAsync(ctx->d_jcoef, 0, ctx->jcoef_cap * sizeof(int16_t), ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream)); // once per (re)allocation: the first decode may run on another stream
        }
    }
    if (!rc) rc = jpeg_grow(ctx, &ctx->d_jsamples, &ctx->jsamples_cap, nblocks * 64, blocks_max * 64);
    const size_t nsub_max = (V + 4096) / ctx->jsub_bytes + 2, nsub = file_bytes / ctx->jsub_bytes + 2;
    if (!rc) rc = jpeg_grow(ctx, &ctx->d_jsub, &ctx->jsub_cap, nsub * 24 + 64, nsub_max * 24 + 64); // + the flag / barrier words
    const size_t desc = sizeof(JpegDev) + 4 * nint, desc_max = sizeof(JpegDev) + 4 * (V / 64 + side / 8 + 64);
    if (!rc) rc = jpeg_grow(ctx, (uint8_t **)&ctx->d_jdev, &ctx->jdev_cap, desc, desc_max);
    if (!rc && ctx->hjdesc_cap < desc) {
        if (ctx->h_jdesc) {
            if (ctx->ev_jdesc) CK(cudaEventSynchronize(ctx->ev_jdesc));
            cudaFreeHost(ctx->h_jdesc); ctx->h_jdesc = nullptr; ctx->hjdesc_cap = 0;
        }
        const size_t want = desc > desc_max ? desc : desc_max;
        CK(cudaMallocHost((void **)&ctx->h_jdesc, want));
        ctx->hjdesc_cap = want;
    }
    if (!rc && !ctx->d_jerr) { CK(cudaMalloc((void **)&ctx->d_jerr, 2 * sizeof(uint32_t))); CK(cudaMemset(ctx->d_jerr, 0, 2 * sizeof(uint32_t))); }
    if (!rc && !ctx->ev_jdesc) CK(cudaEventCreateWithFlags(&ctx->ev_jdesc, cudaEventDisableTiming));
    if (!rc && !ctx->ev_jdone) CK(cudaEventCreateWithFlags(&ctx->ev_jdone, cudaEventDisableTiming));
    if (!rc && !ctx->jplan && !(ctx->jplan = new (std::nothrow) JpegPlan())) return fail(ctx, GSEG_E_ARG, "out of host memory", cudaSuccess);
    return rc;
}

// Enqueue the decode of a parsed file on stream s: interleaved RGB, tightly packed, into rgb_out (device memory).
// The decoder's buffers belong to the context, so a decode is ordered behind the previous one (whatever its stream).
// The next segmentation of the context hands the decode's error word to its control block.
static int jpeg_decode_enqueue(gseg_ctx *ctx, const uint8_t *file, const JpegPlan &plan, uint8_t *rgb_out, cudaStream_t s) {
    const JpegDev &d = plan.dev;
    const uint32_t base = d.data_off & ~15u; // the entropy-coded segment is all the device needs
    const size_t nbytes = (size_t)d.data_end - base;
    int rc = jpeg_reserve_own(ctx, nbytes, (size_t)d.nint, (size_t)d.nblocks);
    if (rc) return rc;
    // the descriptor (offsets relative to the staged bytes) goes through the context's pinned buffer; the restart
    // intervals' start offsets are found on the device (k_jpeg_scan) -- the host never walks the compressed data
    CK(cudaEventSynchronize(ctx->ev_jdesc)); // the previous image's copy out of this buffer
    JpegDev *hd = (JpegDev *)ctx->h_jdesc;
    *hd = d;
    hd->data_off -= base; hd->data_end -= base;
    CK(cudaStreamWaitEvent(s, ctx->ev_jdone, 0));
    CK(cudaMemcpyAsync(ctx->d_jdev, ctx->h_jdesc, sizeof(JpegDev), cudaMemcpyHostToDevice, s));
    CK(cudaEventRecord(ctx->ev_jdesc, s));
    CK(cudaMemcpyAsync(ctx->d_jfile, file + base, nbytes, cudaMemcpyHostToDevice, s));
    const int slot = ctx->jerr_next;
    ctx->jerr_next ^= 1;
    uint32_t *d_starts = (uint32_t *)((uint8_t *)ctx->d_jdev + sizeof(JpegDev));
    const uint32_t S = ctx->jsub_bytes;
    const size_t nsub = (nbytes - (d.data_off - base) + S - 1) / S;
    if ((d.nint == 1 || d.ri > GSEG_JPEG_SYNC_MIN_RI) && nsub >= 2) {
        // no restart markers, or long intervals (every marker is one more point of re-synchronisation): self-synchronising
        // sub-sequences, one cluster (k_jpeg_sync), then the DC prefix sums
        uint64_t *entryS = (uint64_t *)ctx->d_jsub, *exitS = entryS + nsub;
        uint32_t *nblk = (uint32_t *)(exitS + nsub), *blk0 = nblk + nsub, *flags = blk0 + nsub;
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute at[1];
        const int cs = (int)((nsub + JPG_NT_SYNC - 1) / JPG_NT_SYNC);
        cfg.gridDim = dim3(cs < 1 ? 1 : (cs > 8 ? 8 : cs)); cfg.blockDim = dim3(JPG_NT_SYNC); cfg.dynamicSmemBytes = 0; cfg.stream = s;
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cfg.gridDim.x; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        ctx->launches += 4;
        if (ctx->jsync_grid) { // small blocks + software grid barrier (every block must become resident: at most 2 per SM)
            int gs = (int)((nsub + JPG_NT_GRID - 1) / JPG_NT_GRID);
            if (gs > 2 * ctx->num_sms) gs = 2 * ctx->num_sms;
            CK(cudaMemsetAsync(flags, 0, 5 * sizeof(uint32_t), s));
            k_jpeg_sync_grid<<<gs, JPG_NT_GRID, 0, s>>>(ctx->d_jdev, ctx->d_jfile, entryS, exitS, nblk, blk0, flags, ctx->d_jcoef, ctx->d_jerr + slot, S);
        } else {
            CK(cudaLaunchKernelEx(&cfg, k_jpeg_sync, (const JpegDev *)ctx->d_jdev, (const uint8_t *)ctx->d_jfile, entryS, exitS, nblk, blk0,
                                  flags, ctx->d_jcoef, ctx->d_jerr + slot, S));
        }
        k_jpeg_dcscan<<<d.ncomp, JPG_NT_SYNC, 0, s>>>(ctx->d_jdev, ctx->d_jcoef);
    } else {
        ctx->launches += 4;
        k_jpeg_scan<<<1, JPG_NT_SCAN, 0, s>>>(ctx->d_jdev, ctx->d_jfile, d_starts, ctx->d_jerr + slot);
        k_jpeg_huff<<<(d.nint + JPG_NT_HUFF - 1) / JPG_NT_HUFF, JPG_NT_HUFF, 0, s>>>(ctx->d_jdev, d_starts, ctx->d_jfile, ctx->d_jcoef, ctx->d_jerr + slot);
    }
    k_jpeg_idct<<<(d.nblocks + JPG_NT - 1) / JPG_NT, JPG_NT, 0, s>>>(ctx->d_jdev, ctx->d_jcoef, ctx->d_jsamples);
    const size_t groups = (size_t)((d.w + 7) / 8) * d.h;
    k_jpeg_rgb<<<(unsigned)((groups + JPG_NT - 1) / JPG_NT), JPG_NT, 0, s>>>(ctx->d_jdev, ctx->d_jsamples, rgb_out);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev_jdone, s));
    ctx->jflag_slot = slot;
    return GSEG_OK;
}

// Decode into d_rgb and enqueue the segmentation behind it, all on the context's stream.
static int jpeg_own_async(gseg_ctx *ctx, const uint8_t *file, const JpegPlan &plan, const gseg_params *p) {
    const JpegDev &d = plan.dev;
    if ((size_t)d.w * d.h > ctx->Vmax) return fail(ctx, GSEG_E_SIZE, "image exceeds context capacity", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    ctx->valid = false;
    int rc = jpeg_decode_enqueue(ctx, file, plan, ctx->d_rgb, ctx->stream);
    if (!rc) rc = gseg_segment_async(ctx, ctx->d_rgb, d.w, d.h, 3 * d.w, GSEG_MEM_DEVICE, p);
    if (!rc) ctx->jpeg_used = GSEG_JPEG_OWN;
    return rc;
}

// The decode alone, into caller-owned device memory on a caller-chosen stream (the batch pipeline decodes the next
// image of a context on its copy stream while the context's current image is still being segmented).  In-house decoder
// only: GSEG_E_UNSUPPORTED for files that need nvJPEG under the context's backend setting.
extern "C" int gseg_jpeg_decode_async(gseg_ctx *ctx, const void *jpeg, size_t nbytes, uint8_t *rgb_out_device, size_t out_capacity,
                                      void *cuda_stream, int *w, int *h) {
    if (!ctx || !jpeg || !nbytes || !rgb_out_device) return GSEG_E_ARG;
    if (!ctx->jplan && !(ctx->jplan = new (std::nothrow) JpegPlan())) return fail(ctx, GSEG_E_ARG, "out of host memory", cudaSuccess);
    JpegPlan &plan = *ctx->jplan;
    const int prc = jpeg_parse((const uint8_t *)jpeg, nbytes, plan, false);
    if (prc == JPG_NOT_JPEG) { snprintf(ctx->err, sizeof(ctx->err), "not a JPEG: %s", plan.why); return GSEG_E_ARG; }
    if (prc != JPG_OK) { snprintf(ctx->err, sizeof(ctx->err), "in-house JPEG decoder: %s", plan.why); return GSEG_E_UNSUPPORTED; }
    if (w) *w = plan.dev.w;
    if (h) *h = plan.dev.h;
    if (ctx->jpeg_backend == GSEG_JPEG_NVJPEG) return fail(ctx, GSEG_E_UNSUPPORTED, "this file goes to nvJPEG under the context's backend setting", cudaSuccess);
    if ((size_t)3 * plan.dev.w * plan.dev.h > out_capacity) return fail(ctx, GSEG_E_RANGE, "output buffer too small for the decoded image", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    const int rc = jpeg_decode_enqueue(ctx, (const uint8_t *)jpeg, plan, rgb_out_device, cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream);
    if (!rc) ctx->jpeg_used = GSEG_JPEG_OWN;
    return rc;
}

// Decode with nvJPEG (CUDA toolkit library, dlopen): files the in-house decoder does not take.
static int jpeg_nvjpeg_async(gseg_ctx *ctx, const void *jpeg, size_t nbytes, const gseg_params *p, int *w, int *h) {
    NvJpegApi *a = nvjpeg_api();
    if (!a) return fail(ctx, GSEG_E_UNSUPPORTED, "libnvjpeg.so.12 could not be loaded", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    if (!ctx->jpg_handle) {
        if (a->create(&ctx->jpg_handle) != NVJPEG_STATUS_SUCCESS) { ctx->jpg_handle = nullptr; return fail(ctx, GSEG_E_CUDA, "nvjpegCreateSimple", cudaSuccess); }
        if (a->state_create(ctx->jpg_handle, &ctx->jpg_state) != NVJPEG_STATUS_SUCCESS) {
            a->destroy(ctx->jpg_handle); // no half-built pair: the next call starts over
            ctx->jpg_handle = nullptr; ctx->jpg_state = nullptr;
            return fail(ctx, GSEG_E_CUDA, "nvjpegJpegStateCreate", cudaSuccess);
        }
    }
    int iw = 0, ih = 0;
    if (jpeg_size(a, ctx->jpg_handle, jpeg, nbytes, &iw, &ih)) return fail(ctx, GSEG_E_ARG, "not a JPEG nvJPEG can parse", cudaSuccess);
    if (w) *w = iw;
    if (h) *h = ih;
    if ((size_t)iw * ih > ctx->Vmax) return fail(ctx, GSEG_E_SIZE, "image exceeds context capacity", cudaSuccess);
    nvjpegImage_t out = {};
    out.channel[0] = ctx->d_rgb; out.pitch[0] = (size_t)3 * iw; // interleaved RGB, tightly packed
    ctx->valid = false;
    if (a->decode(ctx->jpg_handle, ctx->jpg_state, (const unsigned char *)jpeg, nbytes, NVJPEG_OUTPUT_RGBI, &out, ctx->stream) != NVJPEG_STATUS_SUCCESS)
        return fail(ctx, GSEG_E_ARG, "nvjpegDecode failed (unsupported or corrupt JPEG)", cudaSuccess);
    const int rc = gseg_segment_async(ctx, ctx->d_rgb, iw, ih, 3 * iw, GSEG_MEM_DEVICE, p); // same stream: ordered after the decode
    if (!rc) ctx->jpeg_used = GSEG_JPEG_NVJPEG;
    return rc;
}

// Which decoder: the in-house kernels take every baseline / extended-sequential Huffman file (gseg_jpeg_core.h) -- one
// thread per restart interval when the intervals are short, self-synchronising sub-sequences otherwise; nvJPEG gets
// what they do not decode (progressive, arithmetic, CMYK ...).
extern "C" int gseg_segment_jpeg_async(gseg_ctx *ctx, const void *jpeg, size_t nbytes, const gseg_params *p, int *w, int *h) {
    if (!ctx || !jpeg || !nbytes || !p) return GSEG_E_ARG;
    if (ctx->pending) return fail(ctx, GSEG_E_STATE, "previous run not waited for", cudaSuccess);
    if (!ctx->jplan && !(ctx->jplan = new (std::nothrow) JpegPlan())) return fail(ctx, GSEG_E_ARG, "out of host memory", cudaSuccess);
    JpegPlan &plan = *ctx->jplan;
    const int prc = jpeg_parse((const uint8_t *)jpeg, nbytes, plan, false);
    if (prc == JPG_NOT_JPEG) { snprintf(ctx->err, sizeof(ctx->err), "not a JPEG: %s", plan.why); return GSEG_E_ARG; }
    if (prc == JPG_OK) {
        if (w) *w = plan.dev.w;
        if (h) *h = plan.dev.h;
    }
    const bool own = prc == JPG_OK && ctx->jpeg_backend != GSEG_JPEG_NVJPEG;
    if (ctx->jpeg_backend == GSEG_JPEG_OWN && prc != JPG_OK) {
        snprintf(ctx->err, sizeof(ctx->err), "in-house JPEG decoder: %s", plan.why);
        return GSEG_E_UNSUPPORTED;
    }
    if (own) return jpeg_own_async(ctx, (const uint8_t *)jpeg, plan, p);
    return jpeg_nvjpeg_async(ctx, jpeg, nbytes, p, w, h);
}
extern "C" int gseg_set_jpeg_backend(gseg_ctx *ctx, int backend) {
    if (!ctx || backend < GSEG_JPEG_AUTO || backend > GSEG_JPEG_NVJPEG) return GSEG_E_ARG;
    ctx->jpeg_backend = backend;
    return GSEG_OK;
}
extern "C" int gseg_jpeg_backend_used(const gseg_ctx *ctx) { return ctx ? ctx->jpeg_used : GSEG_E_ARG; }
extern "C" int gseg_segment_jpeg(gseg_ctx *ctx, const void *jpeg, size_t nbytes, const gseg_params *p, int *w, int *h) {
    const int rc = gseg_segment_jpeg_async(ctx, jpeg, nbytes, p, w, h);
    return rc ? rc : gseg_wait(ctx);
}
extern "C" int gseg_input_rgb(gseg_ctx *ctx, uint8_t *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (ctx->pending) { const int rc = gseg_wait(ctx); if (rc) return rc; }
    if (!ctx->valid || !ctx->rgb_staged) return fail(ctx, GSEG_E_STATE, "the last run's input was not staged by the context", cudaSuccess);
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return fail(ctx, GSEG_E_ARG, "mem_kind", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->d_rgb + (size_t)3 * ctx->w * ctx->halo_top, (size_t)3 * ctx->w * ctx->h,
                       mem_kind == GSEG_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

extern "C" void gseg_destroy(gseg_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    cudaFree(ctx->d_rgb); cudaFree(ctx->d_tmp); cudaFree(ctx->d_planes);
    cudaFree(ctx->d_G); cudaFree(ctx->d_wgrid); cudaFree(ctx->d_wsel);
    cudaFree(ctx->d_succ); cudaFree(ctx->d_rank);
    for (int i = 0; i < 2; ++i) {
        cudaFree(ctx->d_best[i]); cudaFree(ctx->d_attr[i]); cudaFree(ctx->d_csum[i]); cudaFree(ctx->d_cmean[i]);
        cudaFree(ctx->d_eab[i]); cudaFree(ctx->d_ew[i]); cudaFree(ctx->d_pcnt[i]); cudaFree(ctx->d_poff[i]); cudaFree(ctx->d_labels[i]);
    }
    cudaFree(ctx->d_pscan); cudaFree(ctx->d_arena); cudaFree(ctx->d_statusC); cudaFree(ctx->d_statusE); cudaFree(ctx->d_ctl);
    jpeg_release(ctx);
    cudaFree(ctx->d_jfile); cudaFree(ctx->d_jsamples); cudaFree(ctx->d_jdev); cudaFree(ctx->d_jcoef);
    if (ctx->h_jdesc) cudaFreeHost(ctx->h_jdesc);
    cudaFree(ctx->d_jerr); cudaFree(ctx->d_jsub);
    if (ctx->ev_jdesc) cudaEventDestroy(ctx->ev_jdesc);
    if (ctx->ev_jdone) cudaEventDestroy(ctx->ev_jdone);
    delete ctx->jplan;
    sort_scratch_free(&ctx->sort);
    cudaFree(ctx->d_xkeys); cudaFree(ctx->d_xvals); cudaFree(ctx->d_xkeep); cudaFree(ctx->d_xab); cudaFree(ctx->d_xw);
    cudaFree(ctx->d_winner); cudaFree(ctx->d_dd); cudaFree(ctx->d_rtab);
    for (int i = 0; i <= GSEG_MAXMARK; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->h_ctl) cudaFreeHost(ctx->h_ctl);
    if (ctx->h_head) cudaFreeHost(ctx->h_head);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    free(ctx);
}

extern "C" int gseg_set_stream(gseg_ctx *ctx, void *s) {
    if (!ctx) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return GSEG_OK;
}

extern "C" int gseg_tail_cluster(const gseg_ctx *ctx) { return ctx ? ctx->tail_cluster : GSEG_E_ARG; }
extern "C" int gseg_tail_cluster_from_env(const gseg_ctx *ctx) { return ctx && ctx->tail_cluster_env ? 1 : 0; }
extern "C" void *gseg_get_stream(const gseg_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

extern "C" int gseg_set_tail(gseg_ctx *ctx, uint32_t max_edges, uint32_t max_components) {
    if (!ctx) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    ctx->tail_E = max_edges; ctx->tail_V = max_components;
    ctx->nbig_hint = -1;
    return GSEG_OK;
}

extern "C" int gseg_set_dedup(gseg_ctx *ctx, int on, uint32_t min_edges, uint32_t min_ratio, uint32_t max_components) {
    if (!ctx) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    ctx->dd_on = on != 0;
    if (min_edges) ctx->dd_min_edges = min_edges;
    if (min_ratio) ctx->dd_min_ratio = min_ratio;
    if (max_components) ctx->dd_V = max_components;
    ctx->nbig_hint = -1; ctx->dd_skip = false;
    CK(upload_dd(ctx));
    return GSEG_OK;
}

extern "C" int gseg_set_tail_cluster(gseg_ctx *ctx, int ctas) {
    if (!ctx || ctas < 1 || ctas > 16) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    ctx->tail_cluster = fit_tail_cluster(ctas);
    return GSEG_OK;
}

extern "C" int gseg_set_blocks_per_sm(gseg_ctx *ctx, int blocks) {
    if (!ctx || blocks < 1 || blocks > 8) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    ctx->occ_mult = blocks;
    return GSEG_OK;
}

// Gaussian taps (same definition as the oracle's orc_gauss_mask; double arithmetic, one final rounding).
static int gauss_mask(float sigma, float *mask) {
    if (sigma < 0.01f) sigma = 0.01f;
    const int len = (int)ceilf(sigma * 4.0f) + 1;
    if (len > GSEG_MAXMASK) return -1;
    double m[GSEG_MAXMASK], s = 0.0;
    for (int i = 0; i < len; ++i) {
        const double t = (double)i / (double)sigma;
        m[i] = exp(-0.5 * t * t);
    }
    for (int i = 1; i < len; ++i) s += m[i];
    s = 2.0 * s + m[0];
    for (int i = 0; i < len; ++i) mask[i] = (float)(m[i] / s);
    return len;
}

// Called right before every kernel launch: counts it and, when profiling, drops an event so that
// consecutive events bracket exactly one kernel.
static inline void mark(gseg_ctx *c, cudaStream_t s, const char *name, int round) {
    ++c->launches;
    if (!c->profiling || c->n_marks >= GSEG_MAXMARK) return;
    if (!c->ev[c->n_marks]) cudaEventCreate(&c->ev[c->n_marks]);
    cudaEventRecord(c->ev[c->n_marks], s);
    c->mark_name[c->n_marks] = name;
    c->mark_round[c->n_marks] = round;
    ++c->n_marks;
}
// Closes the last kernel of a round before the host read-back gap (a nameless mark).
static inline void mark_end(gseg_ctx *c, cudaStream_t s) {
    if (!c->profiling || c->n_marks == 0 || c->n_marks >= GSEG_MAXMARK) return;
    if (!c->ev[c->n_marks]) cudaEventCreate(&c->ev[c->n_marks]);
    cudaEventRecord(c->ev[c->n_marks], s);
    c->mark_name[c->n_marks] = nullptr;
    c->mark_round[c->n_marks] = -1;
    ++c->n_marks;
}

// ---- round scheduling --------------------------------------------------------------------------
static GsegBufs bufs_of(const gseg_ctx *c) {
    GsegBufs B;
    B.planes = c->d_planes; B.G = c->d_G; B.wgrid = c->d_wgrid;
    B.succ = c->d_succ; B.rank = c->d_rank; B.wsel = c->d_wsel; B.arena = c->d_arena;
    for (int i = 0; i < 2; ++i) {
        B.best[i] = c->d_best[i]; B.attr[i] = c->d_attr[i]; B.csum[i] = c->d_csum[i]; B.cmean[i] = c->d_cmean[i];
        B.eab[i] = c->d_eab[i]; B.ew[i] = c->d_ew[i]; B.pcnt[i] = c->d_pcnt[i]; B.poff[i] = c->d_poff[i];
    }
    B.statusC = c->d_statusC; B.statusE = c->d_statusE; B.pscan = c->d_pscan;
    return B;
}

template <int R>
static size_t blur_smem() { return (size_t)3 * (TH + 2 * R) * (BLUR_PF(R) + BLUR_PH * sizeof(float)); } // 8-bit staged input + fp32 horizontal pass
template <int R>
static void launch_blur(gseg_ctx *c, cudaStream_t s, int ntiles) {
    static bool attr[64] = {false}; // the opt-in is per function and per device
    if (!attr[c->device & 63]) { cudaFuncSetAttribute(k_blur_tile<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)blur_smem<R>()); attr[c->device & 63] = true; }
    k_blur_tile<R><<<ntiles, NT, blur_smem<R>(), s>>>(c->d_ctl, c->d_planes);
}

template <int VARIANT, int D>
static size_t graph_smem() {
    return (size_t)(3 + D + (VARIANT == GSEG_SUPERPIX ? 1 : 0)) * BH * BW * sizeof(float) + 16; // the choice bytes reuse the colour planes
}
template <int VARIANT, int D>
static void launch_r0_graph(gseg_ctx *c, cudaStream_t s, int ntiles, const GsegBufs &B) {
    static bool attr[64] = {false};
    if (!attr[c->device & 63]) { cudaFuncSetAttribute(k_r0_graph<VARIANT, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)graph_smem<VARIANT, D>()); attr[c->device & 63] = true; }
    k_r0_graph<VARIANT, D><<<ntiles < c->num_sms * c->occ_mult ? ntiles : c->num_sms * c->occ_mult, NT, graph_smem<VARIANT, D>(), s>>>(c->d_ctl, B);
}
template <int D, bool SP>
static void launch_r0_edges(gseg_ctx *c, cudaStream_t s, size_t V, const GsegBufs &B) {
    static bool attr[64] = {false};
    if (!attr[c->device & 63]) { cudaFuncSetAttribute(k_r0_edges<D, SP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R0_SMEM); attr[c->device & 63] = true; }
    const size_t pages = (size_t)D * ((V + GSEG_PAGE - 1) / GSEG_PAGE);
    const size_t ntiles = (pages + NT / 32 - 1) / (NT / 32); // blocks that cover all pages
    const int grid = (int)(ntiles < (size_t)c->num_sms * c->occ_mult ? ntiles : (size_t)c->num_sms * c->occ_mult);
    // profiled as k_r0_edges (staged body) or k_r0_edges_rl (register-load body)
    if (pages <= (size_t)c->r0_stage_ppw * grid * (NT / 32)) {
        mark(c, s, "k_r0_edges", 0);
        k_r0_edges<D, SP, true><<<grid, NT, R0_SMEM, s>>>(c->d_ctl, B);
    } else {
        mark(c, s, "k_r0_edges_rl", 0);
        k_r0_edges<D, SP, false><<<grid, NT, 0, s>>>(c->d_ctl, B);
    }
}

// Round 0: blur -> [sobel] -> fused graph kernel -> relabel -> edge list.  4-5 launches.
static void enqueue_round0(gseg_ctx *c, cudaStream_t s) {
    const size_t V = (size_t)c->w * c->h;
    const int variant = c->params.variant, D = c->D;
    const bool sp = variant == GSEG_SUPERPIX;
    const GsegBufs B = bufs_of(c);
    const int ntiles = ((c->w + TW - 1) / TW) * ((c->h + TH - 1) / TH);  // blur tiles
    const int ntilesG = ((c->w + TW - 1) / TW) * ((c->h + GH - 1) / GH); // graph tiles
    const int R = c->h_head->p.mask_len - 1;
    if (R >= 1 && R <= 8) {
        mark(c, s, "k_blur_tile", 0);
        switch (R) {
        case 1: launch_blur<1>(c, s, ntiles); break;
        case 2: launch_blur<2>(c, s, ntiles); break;
        case 3: launch_blur<3>(c, s, ntiles); break;
        case 4: launch_blur<4>(c, s, ntiles); break;
        case 5: launch_blur<5>(c, s, ntiles); break;
        case 6: launch_blur<6>(c, s, ntiles); break;
        case 7: launch_blur<7>(c, s, ntiles); break;
        default: launch_blur<8>(c, s, ntiles); break;
        }
    } else {
        mark(c, s, "k_blur_h", 0);
        k_blur_h<<<grid_for((size_t)c->w * c->h_head->p.h_in, NT), NT, 0, s>>>(c->d_ctl, c->d_tmp);
        mark(c, s, "k_blur_v", 0);
        k_blur_v<<<grid_for(3 * V, NT), NT, 0, s>>>(c->d_ctl, c->d_tmp, c->d_planes);
    }
    if (sp) {
        mark(c, s, "k_sobel", 0);
        k_sobel<<<grid_for(V, NT), NT, 0, s>>>(c->d_ctl, c->d_planes, c->d_G);
    }
    mark(c, s, "k_r0_graph", 0);
    if (variant == GSEG_FELZ) { if (D == 2) launch_r0_graph<GSEG_FELZ, 2>(c, s, ntilesG, B); else launch_r0_graph<GSEG_FELZ, 4>(c, s, ntilesG, B); }
    else if (variant == GSEG_HIER) { if (D == 2) launch_r0_graph<GSEG_HIER, 2>(c, s, ntilesG, B); else launch_r0_graph<GSEG_HIER, 4>(c, s, ntilesG, B); }
    else { if (D == 2) launch_r0_graph<GSEG_SUPERPIX, 2>(c, s, ntilesG, B); else launch_r0_graph<GSEG_SUPERPIX, 4>(c, s, ntilesG, B); }
    mark(c, s, "k_relabel", 0);
    if (sp) k_relabel<true, true><<<grid_for(V, NT), NT, 0, s>>>(c->d_ctl, B);
    else k_relabel<true, false><<<grid_for(V, NT), NT, 0, s>>>(c->d_ctl, B);
    if (sp) {
        mark(c, s, "k_means", 0);
        k_means<<<grid_for(V, NT, c->num_sms * c->occ_mult), NT, 0, s>>>(c->d_ctl, B);
    }
    if (D == 2) { if (sp) launch_r0_edges<2, true>(c, s, V, B); else launch_r0_edges<2, false>(c, s, V, B); }
    else { if (sp) launch_r0_edges<4, true>(c, s, V, B); else launch_r0_edges<4, false>(c, s, V, B); }
}

// One grid-wide round r >= 1: 3 launches.  Vb/Eb bound the round's component / edge counts (exact after
// a read-back in the host-driven schedule, the image's own bounds otherwise); every kernel takes its
// real sizes from the device-resident round state and surplus blocks exit through the tile tickets.
static void enqueue_round(gseg_ctx *c, cudaStream_t s, int r, size_t Vb, size_t Pb) {
    const bool sp = c->params.variant == GSEG_SUPERPIX;
    const GsegBufs B = bufs_of(c);
    const int cap = c->num_sms * c->occ_mult;
    if (Pb > GSEG_PSCAN_INLINE) { // Pb bounds the round's page count: below, the successor kernel's extra block scans
        mark(c, s, "k_page_scan", r);
        k_page_scan<<<grid_for(Pb, 1024, 64), 1024, 0, s>>>(c->d_ctl, B);
    }
    mark(c, s, "k_succ_scan", r);
    if (sp) k_succ_scan<true><<<grid_for(Vb, NT * CPT, cap) + 1, NT, 0, s>>>(c->d_ctl, B);
    else k_succ_scan<false><<<grid_for(Vb, NT * CPT, cap) + 1, NT, 0, s>>>(c->d_ctl, B);
    mark(c, s, "k_relabel", r);
    if (sp) k_relabel<false, true><<<grid_for(Vb, NT, cap), NT, 0, s>>>(c->d_ctl, B);
    else k_relabel<false, false><<<grid_for(Vb, NT, cap), NT, 0, s>>>(c->d_ctl, B);
    if (sp) {
        mark(c, s, "k_means", r);
        k_means<<<grid_for(Vb, NT, cap), NT, 0, s>>>(c->d_ctl, B);
    }
    mark(c, s, "k_edges", r);
    if (sp) k_edges<true><<<grid_for(Pb, NT / 32, cap), NT, 0, s>>>(c->d_ctl, B);
    else k_edges<false><<<grid_for(Pb, NT / 32, cap), NT, 0, s>>>(c->d_ctl, B);
}

// Duplicate elimination between rounds (gseg_dedup.cuh): 11 launches that size themselves from the device-resident
// state and exit at once unless the plan kernel decides to run.  Enqueued in front of every tail launch.
static u32 dedup_V(const gseg_ctx *c) { // components from which on the list is de-duplicated (<= 65536: two ids in a 32-bit key)
    const u32 v = c->dd_V > 2u ? c->dd_V : 2u;
    return v < 65536u ? v : 65536u;
}
static bool dedup_enabled(const gseg_ctx *c) {
    return c->dd_on && c->params.variant != GSEG_SUPERPIX && !(c->params.flags & GSEG_FLAG_NO_DEDUP);
}
// Device-driven schedule: the sequence is enqueued blind.  Once an image of this shape has shown that it never meets the
// thresholds, its eleven self-skipping launches are left out for the following images of the same shape.
static bool dedup_enqueue(const gseg_ctx *c) {
    return dedup_enabled(c) &&
           !(c->dd_skip && c->hint_w == c->w && c->hint_h == c->h && c->hint_variant == c->params.variant && c->hint_conn == c->params.connectivity);
}
static void enqueue_dedup(gseg_ctx *c, cudaStream_t s, int round) {
    const GsegBufs B = bufs_of(c);
    const int cap = c->num_sms * c->occ_mult;
    const size_t ntiles = (c->dd_cap + SORT_TILE - 1) / SORT_TILE;
    const int gs = (int)(ntiles < (size_t)c->num_sms * 2 ? ntiles : (size_t)c->num_sms * 2);
    mark(c, s, "k_dd_plan", round);
    k_dd_plan<<<1, 1024, 0, s>>>(c->d_ctl, B, c->d_dd);
    mark(c, s, "k_dd_keys", round);
    k_dd_keys<<<cap, NT, 0, s>>>(c->d_ctl, B, c->d_dd);
    mark(c, s, "k_sort_scan", round);
    k_sort_scan_dev<<<4, SORT_RADIX, 0, s>>>(&c->d_dd->sort);
    for (int p = 0; p < 4; ++p) { // two ids of <= 16 bits each: at most four 8-bit passes
        mark(c, s, "k_sort_onesweep", round);
        k_sort_onesweep_dev<<<gs, SORT_NT, sort_smem_bytes(), s>>>(&c->d_dd->sort, p);
    }
    mark(c, s, "k_dd_select", round);
    k_dd_select<<<cap, NT, 0, s>>>(c->d_dd);
    mark(c, s, "k_dd_mark", round);
    k_dd_mark<<<cap, NT, 0, s>>>(c->d_ctl, B, c->d_dd);
    mark(c, s, "k_dd_compact", round);
    k_dd_compact<<<grid_for(c->dd_cap, 4096, c->num_sms * 2), 1024, 0, s>>>(c->d_ctl, B, c->d_dd);
    mark(c, s, "k_dd_finish", round);
    k_dd_finish<<<cap, NT, 0, s>>>(c->d_ctl, B, c->d_dd);
}
// Host-driven schedule: the same decision as k_dd_plan, from the state just read back (so that the profiled schedule
// only launches the sequence when it runs).
static bool dedup_wanted_host(const gseg_ctx *c) {
    const RoundState &st = c->h_ctl->st;
    return dedup_enabled(c) && st.phase != PH_DONE && st.round >= 1u && st.V >= 2u && st.V <= dedup_V(c) && st.E <= c->dd_cap &&
           st.E >= c->dd_min_edges && st.E / st.V >= c->dd_min_ratio;
}

// The tail: one cluster runs every remaining (small) round.
static cudaError_t enqueue_tail(gseg_ctx *c, cudaStream_t s) {
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[1];
    cfg.gridDim = dim3(c->tail_cluster); cfg.blockDim = dim3(NTT);
    cfg.dynamicSmemBytes = TAIL_SMEM; cfg.stream = s;
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = c->tail_cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    GsegCtl *ctl = c->d_ctl;
    GsegBufs B = bufs_of(c);
    mark(c, s, "k_tail", -1);
    if (c->params.variant == GSEG_SUPERPIX) return cudaLaunchKernelEx(&cfg, k_tail<true>, ctl, B);
    return cudaLaunchKernelEx(&cfg, k_tail<false>, ctl, B);
}

static size_t edge_slots(const gseg_ctx *ctx) {
    return (size_t)ctx->Dmax * ((ctx->Vmax + GSEG_PAGE - 1) / GSEG_PAGE + 1) * GSEG_PAGE;
}

static int max_rounds_of(const gseg_params *p) {
    int r = p->max_rounds > 0 ? p->max_rounds : 48;
    return r > GSEG_MAXR ? GSEG_MAXR : r;
}

static int readback(gseg_ctx *ctx) {
    CK(cudaMemcpyAsync(ctx->h_ctl, ctx->d_ctl, sizeof(GsegCtl), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

static int finish(gseg_ctx *ctx) {
    ctx->pending = false;
    if (ctx->h_ctl->error == DERR_SCAN) return fail(ctx, GSEG_E_INTERNAL, "look-back watchdog", cudaSuccess);
    if (ctx->h_ctl->error == DERR_ARENA) return fail(ctx, GSEG_E_ARENA, "map arena", cudaSuccess);
    if (ctx->h_ctl->error == DERR_CHASE) return fail(ctx, GSEG_E_INTERNAL, "successor cycle", cudaSuccess);
    if (ctx->h_ctl->error == DERR_JPEG) return fail(ctx, GSEG_E_ARG, "corrupt JPEG: the entropy-coded data does not decode", cudaSuccess);
    if (ctx->h_ctl->error >= DERR_CHECK) {
        snprintf(ctx->err, sizeof(ctx->err), "checked build: bounds check at site %u failed", ctx->h_ctl->error - DERR_CHECK);
        return GSEG_E_INTERNAL;
    }
    // remember how many grid-wide rounds this kind of image needed before the tail could take over, and whether the
    // duplicate elimination ever ran (device-driven runs only: a host-driven run has no tail and decides per round)
    const GsegCtl *h = ctx->h_ctl;
    if (!(ctx->params.flags & GSEG_FLAG_HOST_LOOP)) {
        int nbig = 0;
        bool ran = false;
        for (u32 r = 1; r < h->st.round; ++r) {
            if (!h->stTail[r]) nbig = (int)r;
            ran = ran || h->stDedupOut[r] != 0u;
        }
        ctx->nbig_hint = nbig;
        ctx->dd_skip = dedup_enabled(ctx) && !ran;
        ctx->hint_w = ctx->w; ctx->hint_h = ctx->h; ctx->hint_variant = ctx->params.variant; ctx->hint_conn = ctx->params.connectivity;
    }
    ctx->valid = true;
    return GSEG_OK;
}

// Arena compaction (FELZ and explicit-graph FELZ runs only: they need the final partition, not the levels).
// The device stopped because the next round's map does not fit (error = DERR_ARENA, resume_phase = the phase
// to go on with).  Fold the stored maps into one and resume:
//   A: the maps of all live rounds f..r (f = first live round >= 1) into round f's slot;
//   B: if that does not free enough, everything into round 0's pixel map, in place.
// Returns 1 when the run can go on, 0 when nothing could be freed (a genuine GSEG_E_ARENA), < 0 on CUDA errors.
static int compact_arena(gseg_ctx *ctx) {
    GsegCtl *h = ctx->h_ctl;
    if (ctx->params.variant != GSEG_FELZ || h->resume_phase == PH_DONE) return 0;
    const int rn = (int)h->st.round;          // the round that could not start
    const int r0 = ctx->graph_mode ? 1 : 0;   // first round that stored a map
    const u64 cap = ctx->arena_cap, Vn = h->st.V;
    int f = -1, live = 0;
    for (int r = r0 + 1; r < rn; ++r)
        if (!h->map_skip[r]) { if (f < 0) f = r; ++live; }
    cudaStream_t s = ctx->stream;
    bool done = false;
    if (live >= 2 && (u64)h->map_off[f] + h->stV[f] + Vn <= cap) { // A
        const u32 n = h->stV[f];
        ctx->launches += 1;
        k_compose_table<<<grid_for(n, NT), NT, 0, s>>>(ctx->d_ctl, ctx->d_arena, f, rn - 1, n, ctx->d_wsel); // wsel is dead between rounds
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(ctx->d_arena + h->map_off[f], ctx->d_wsel, (size_t)n * sizeof(u32), cudaMemcpyDeviceToDevice, s));
        for (int r = f + 1; r < rn; ++r) h->map_skip[r] = 1;
        h->st.map_off = h->map_off[f] + n;
        done = true;
    } else if (!ctx->graph_mode && live >= 1 && (u64)h->stV[0] + Vn <= cap) { // B
        ctx->launches += 1;
        k_compose_inplace<<<grid_for(h->stV[0], NT), NT, 0, s>>>(ctx->d_ctl, ctx->d_arena, rn - 1);
        CK(cudaGetLastError());
        for (int r = 1; r < rn; ++r) h->map_skip[r] = 1;
        h->st.map_off = h->stV[0];
        done = true;
    }
    if (!done) return 0;
    h->map_off[rn] = h->st.map_off;
    h->st.phase = h->resume_phase; h->resume_phase = PH_DONE; h->error = DERR_NONE;
    // the device is idle (the read-back synchronised) and h is its exact image: write the patched block back
    CK(cudaMemcpyAsync(ctx->d_ctl, h, sizeof(GsegCtl), cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s)); // h is about to be overwritten by the next read-back
    ++ctx->compactions;
    return 1;
}

// After a read-back: does the run have to go on?  (Handles the arena compaction.)  < 0 on errors.
static int run_continues(gseg_ctx *ctx) {
    if (ctx->h_ctl->error == DERR_ARENA) return compact_arena(ctx);
    return ctx->h_ctl->st.phase != PH_DONE && ctx->h_ctl->error == DERR_NONE ? 1 : 0;
}

// Buffers only some paths need: d_tmp (blur with more than 8 taps), d_G + d_csum + d_cmean (superpixel),
// d_labels[1] (all-levels / colour images to host memory).  gseg_reserve allocates them up front; without
// it they are allocated by the first call that needs them (an allocation synchronises the device).
template <typename T>
static int ensure(gseg_ctx *ctx, T **p, size_t n) {
    if (*p) return GSEG_OK;
    CK(dalloc(p, n));
    return GSEG_OK;
}

static int ensure_csum(gseg_ctx *ctx) {
    if (ctx->d_csum[0] && ctx->d_csum[1] && ctx->d_cmean[0] && ctx->d_cmean[1]) return GSEG_OK;
    for (int i = 0; i < 2; ++i) {
        int rc = ensure(ctx, &ctx->d_csum[i], 3 * (ctx->Vmax + 64));
        if (!rc) rc = ensure(ctx, &ctx->d_cmean[i], ctx->Vmax + 64);
        if (rc) return rc;
    }
    return GSEG_OK;
}

extern "C" int gseg_reserve(gseg_ctx *ctx, uint32_t caps) {
    if (!ctx || (caps & ~(GSEG_CAP_SUPERPIX | GSEG_CAP_WIDE_SIGMA | GSEG_CAP_LEVELS | GSEG_CAP_JPEG | GSEG_CAP_REGIONS))) return GSEG_E_ARG;
    if (ctx->pending) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    int rc = GSEG_OK;
    if (caps & GSEG_CAP_SUPERPIX) { rc = ensure_csum(ctx); if (!rc) rc = ensure(ctx, &ctx->d_G, ctx->Vmax + 64); }
    if (!rc && (caps & GSEG_CAP_WIDE_SIGMA)) rc = ensure(ctx, &ctx->d_tmp, 3 * (ctx->Vmax + 64));
    if (!rc && (caps & GSEG_CAP_LEVELS)) rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64);
    if (!rc && (caps & GSEG_CAP_JPEG)) rc = jpeg_reserve_own(ctx, 0, 0, 0);
    if (!rc && (caps & GSEG_CAP_REGIONS)) {
        rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64);
        if (!rc) rc = ensure(ctx, &ctx->d_rtab, 8 * (ctx->Vmax + 64));
    }
    return rc;
}

extern "C" void *gseg_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (!bytes || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void *gseg_host_alloc_wc(size_t bytes) {
    void *p = nullptr;
    if (!bytes || cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocWriteCombined) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void gseg_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

// Grid-wide rounds to enqueue ahead of the tail when nothing is known about the image: live edges
// shrink by roughly 0.55-0.6x per round on natural and synthetic images (Report.pdf p5: 10-20 rounds).
static int estimate_nbig(const gseg_ctx *c) {
    double E = 0.62 * (double)c->w * c->h * c->D, V = 0.3 * (double)c->w * c->h;
    int n = 0;
    // with the duplicate elimination in front of the tail, the tail takes over as soon as V <= tail_V (the list then
    // shrinks to ~3 V edges); without it, when the list itself has shrunk to tail_E
    const bool dd = dedup_enqueue(c);
    while ((V > c->tail_V || E > c->tail_E) && !(dd && V <= dedup_V(c) && E >= c->dd_min_edges) && n < GSEG_MAXR) { E *= 0.6; V *= 0.27; ++n; }
    return n;
}

// The image this run reads was decoded by the in-house JPEG decoder: its error word goes to the control block, behind
// every kernel of the run and in front of gseg_wait's read-back.
static cudaError_t jpeg_flag_enqueue(gseg_ctx *ctx, int slot) {
    if (slot < 0) return cudaSuccess;
    k_jpeg_flag<<<1, 1, 0, ctx->stream>>>(ctx->d_jerr + slot, ctx->d_ctl);
    ++ctx->launches;
    return cudaGetLastError();
}

// rgb points at the first row of the buffer: halo_top rows of halo, the h rows to segment, halo_bottom rows of halo.
static int segment_async_impl(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride, int mem_kind, int halo_top,
                              int halo_bottom, const gseg_params *p) {
    if (!ctx || !rgb || !p) return GSEG_E_ARG;
    if (ctx->pending) return fail(ctx, GSEG_E_STATE, "previous run not waited for", cudaSuccess);
    const int jslot = ctx->jflag_slot; // this run's input came out of the in-house JPEG decoder (else -1)
    ctx->jflag_slot = -1;
    if (w < 1 || h < 1 || stride < 3 * w || halo_top < 0 || halo_bottom < 0) return fail(ctx, GSEG_E_ARG, "image geometry", cudaSuccess);
    if ((size_t)w * h > ctx->Vmax) return fail(ctx, GSEG_E_SIZE, "image exceeds context capacity", cudaSuccess);
    const int h_in = h + halo_top + halo_bottom;
    if (mem_kind == GSEG_MEM_HOST && (size_t)w * h_in > ctx->Vmax) // host input is staged whole, halo rows included
        return fail(ctx, GSEG_E_SIZE, "strip + halo rows exceed the context's staging capacity", cudaSuccess);
    if ((size_t)((w + TW - 1) / TW) * (size_t)((h + GH - 1) / GH) > ctx->ntilesC)
        return fail(ctx, GSEG_E_SIZE, "image aspect exceeds context capacity", cudaSuccess);
    if (p->connectivity != 4 && p->connectivity != 8) return fail(ctx, GSEG_E_ARG, "connectivity must be 4 or 8", cudaSuccess);
    if (p->variant < GSEG_FELZ || p->variant > GSEG_SUPERPIX) return fail(ctx, GSEG_E_ARG, "variant", cudaSuccess);
    if (!(p->sigma >= 0.0f) || p->max_levels < 0 || p->max_rounds < 0 || p->min_size < 0 || !(p->k >= 0.0f)) return fail(ctx, GSEG_E_ARG, "parameter range", cudaSuccess);
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return fail(ctx, GSEG_E_ARG, "mem_kind", cudaSuccess);
    GsegHead *hh = ctx->h_head;
    GsegRunParams *hp = &hh->p;
    const int len = gauss_mask(p->sigma, hp->mask);
    if (len < 0) return fail(ctx, GSEG_E_ARG, "sigma too large (more than 64 taps)", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    ctx->valid = false; ctx->x_valid = false; ctx->graph_mode = false; ctx->strip_labels = false; ctx->halo_top = halo_top;
    ctx->params = *p;
    ctx->w = w; ctx->h = h; ctx->D = p->connectivity == 8 ? 4 : 2;
    if (ctx->D > ctx->Dmax) return fail(ctx, GSEG_E_SIZE, "context was created for 4-connected grids only", cudaSuccess);
    if (p->variant == GSEG_SUPERPIX) {
        int rc = ensure_csum(ctx);
        if (!rc) rc = ensure(ctx, &ctx->d_G, ctx->Vmax + 64);
        if (rc) return rc;
    }
    if (len - 1 > 8 || len - 1 < 1) {
        if ((size_t)w * h_in > ctx->Vmax) return fail(ctx, GSEG_E_SIZE, "wide-sigma strip + halo rows exceed the context capacity", cudaSuccess);
        int rc = ensure(ctx, &ctx->d_tmp, 3 * (ctx->Vmax + 64));
        if (rc) return rc;
    }
    const uint8_t *src = rgb;
    int dstride = stride;
    if (mem_kind == GSEG_MEM_HOST) {
        if (stride == 3 * w) // tightly packed rows: one linear copy (a pitched copy is issued row by row)
            CK(cudaMemcpyAsync(ctx->d_rgb, rgb, (size_t)3 * w * h_in, cudaMemcpyHostToDevice, ctx->stream));
        else
            CK(cudaMemcpy2DAsync(ctx->d_rgb, (size_t)3 * w, rgb, (size_t)stride, (size_t)3 * w, (size_t)h_in,
                                 cudaMemcpyHostToDevice, ctx->stream));
        src = ctx->d_rgb;
        dstride = 3 * w;
    }
    ctx->rgb_staged = src == ctx->d_rgb;
    const int R = max_rounds_of(p);
    const bool host_loop = (p->flags & GSEG_FLAG_HOST_LOOP) != 0;
    // look-back tags: 2 per round, 30 bits; recycle the tag space long before it wraps
    if (ctx->epoch_next + GSEG_EPOCHS_PER_RUN >= (1u << 30)) {
        CK(cudaMemsetAsync(ctx->d_statusC, 0, ctx->ntilesC * sizeof(u64), ctx->stream));
        CK(cudaMemsetAsync(ctx->d_statusE, 0, ctx->ntilesE * sizeof(u64), ctx->stream));
        ctx->epoch_next = 1;
    }
    hp->rgb = src; hp->w = w; hp->h = h; hp->stride = dstride; hp->D = ctx->D; hp->variant = p->variant;
    hp->h_in = h_in; hp->y_off = halo_top;
    hp->k = p->k; hp->min_size = p->min_size; hp->max_rounds = R;
    hp->max_levels = p->max_levels > 0 ? p->max_levels : INT_MAX;
    hp->arena_cap = (u32)ctx->arena_cap; hp->edge_slots = (u32)edge_slots(ctx);
    hp->epoch_base = ctx->epoch_next;
    hp->mask_len = len;
    hp->filter_shift = ctx->filter_shift;
    hp->tail_E = ctx->run_tail_E = host_loop ? 0u : ctx->tail_E;
    hp->tail_V = ctx->run_tail_V = host_loop ? 0u : ctx->tail_V;
    hp->tail_P = ctx->tail_P;
    hp->no_dedup = dedup_enabled(ctx) ? 0u : 1u; hp->dd_V = dedup_V(ctx);
    ctx->epoch_next += GSEG_EPOCHS_PER_RUN;
    // the whole head of the control block (parameters + round-0 state + tickets) in one copy
    hh->st.V = (u32)((size_t)w * h); hh->st.E = 0; hh->st.round = 0; hh->st.phase = PH_PRED; hh->st.levels = 0; hh->st.map_off = 0; hh->st.P = 0; hh->st.pad = 0;
    hh->Vnext = hh->st.V; hh->error = DERR_NONE; hh->ticketC = 0; hh->ticketE = 0; hh->doneE = 0;
    memset(hh->Eacc, 0, sizeof(hh->Eacc));
    memset(hh->map_skip, 0, sizeof(hh->map_skip)); hh->resume_phase = PH_DONE;
    memset(hh->stDedupIn, 0, sizeof(hh->stDedupIn)); memset(hh->stDedupOut, 0, sizeof(hh->stDedupOut));
    CK(cudaMemcpyAsync(ctx->d_ctl, hh, sizeof(GsegHead), cudaMemcpyHostToDevice, ctx->stream));

    ctx->n_marks = 0;
    enqueue_round0(ctx, ctx->stream);
    CK(cudaGetLastError());
    if (!host_loop) {
        // device-driven schedule: the grid-wide rounds this kind of image is expected to need, then the
        // tail cluster; no host involvement until gseg_wait (which continues the run if the guess was short)
        int nbig = ctx->nbig_hint;
        if (nbig < 0 || ctx->hint_w != w || ctx->hint_h != h || ctx->hint_variant != p->variant ||
            ctx->hint_conn != p->connectivity)
            nbig = estimate_nbig(ctx);
        if (nbig > R - 1) nbig = R - 1;
        const size_t V = (size_t)w * h;
        for (int r = 1; r <= nbig; ++r) enqueue_round(ctx, ctx->stream, r, V, (size_t)ctx->D * (V / GSEG_PAGE + 1));
        if (dedup_enqueue(ctx)) enqueue_dedup(ctx, ctx->stream, -1);
        CK(cudaGetLastError());
        CK(enqueue_tail(ctx, ctx->stream));
        CK(jpeg_flag_enqueue(ctx, jslot));
        ctx->pending = true;
        return GSEG_OK;
    }
    // host-driven schedule: one 2 KB read-back per round decides termination and sizes the next grids
    mark_end(ctx, ctx->stream);
    int rc = readback(ctx);
    if (rc) return rc;
    for (int go; (go = run_continues(ctx)) != 0;) {
        if (go < 0) return go;
        if (dedup_wanted_host(ctx)) {
            enqueue_dedup(ctx, ctx->stream, (int)ctx->h_ctl->st.round);
            mark_end(ctx, ctx->stream);
            CK(cudaGetLastError());
            rc = readback(ctx);
            if (rc) return rc;
        }
        enqueue_round(ctx, ctx->stream, (int)ctx->h_ctl->st.round, ctx->h_ctl->st.V, ctx->h_ctl->st.P);
        mark_end(ctx, ctx->stream);
        CK(cudaGetLastError());
        rc = readback(ctx);
        if (rc) return rc;
    }
    CK(jpeg_flag_enqueue(ctx, jslot));
    ctx->pending = true;
    return GSEG_OK;
}

// Read the control block back; while the run is not finished (the guess of grid-wide rounds was short)
// keep going, two rounds and a tail at a time.
static int wait_rounds(gseg_ctx *ctx) {
    int rc = readback(ctx);
    if (ctx->params.flags & GSEG_FLAG_HOST_LOOP) return rc; // the host loop already ran the rounds to the end
    for (int go; !rc && (go = run_continues(ctx)) != 0;) {
        if (go < 0) return go;
        const int r = (int)ctx->h_ctl->st.round;
        enqueue_round(ctx, ctx->stream, r, ctx->h_ctl->st.V, ctx->h_ctl->st.P);
        enqueue_round(ctx, ctx->stream, r + 1, ctx->h_ctl->st.V, ctx->h_ctl->st.P);
        if (dedup_enqueue(ctx)) enqueue_dedup(ctx, ctx->stream, -1);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = enqueue_tail(ctx, ctx->stream);
        if (e != cudaSuccess) return fail(ctx, GSEG_E_CUDA, "continuation launch", e);
        rc = readback(ctx);
    }
    return rc;
}

extern "C" int gseg_segment_async(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride, int mem_kind,
                                  const gseg_params *p) {
    return segment_async_impl(ctx, rgb, w, h, stride, mem_kind, 0, 0, p);
}

extern "C" int gseg_segment_strip_async(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride, int mem_kind, int halo_top,
                                        int halo_bottom, const gseg_params *p) {
    if (p && p->variant == GSEG_SUPERPIX) // the Sobel plane would need a halo of blurred rows
        return fail(ctx, GSEG_E_ARG, "strips: FELZ or HIER", cudaSuccess);
    return segment_async_impl(ctx, rgb, w, h, stride, mem_kind, halo_top, halo_bottom, p);
}

extern "C" int gseg_wait(gseg_ctx *ctx) {
    if (!ctx) return GSEG_E_ARG;
    if (!ctx->pending) return ctx->valid ? GSEG_OK : GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    int rc = wait_rounds(ctx);
    if (rc) { ctx->pending = false; return rc; }
    return finish(ctx);
}

extern "C" int gseg_segment(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride, int mem_kind,
                            const gseg_params *p) {
    int rc = gseg_segment_async(ctx, rgb, w, h, stride, mem_kind, p);
    if (rc) return rc;
    return gseg_wait(ctx);
}

extern "C" int gseg_num_levels(const gseg_ctx *ctx) {
    if (!ctx || !ctx->valid) return GSEG_E_STATE;
    return ctx->params.variant == GSEG_FELZ ? 1 : (int)ctx->h_ctl->st.levels;
}

extern "C" int gseg_num_components(const gseg_ctx *ctx, int level) {
    if (!ctx || !ctx->valid) return GSEG_E_STATE;
    const int nl = gseg_num_levels(ctx);
    if (level < 0) level = nl - 1;
    if (ctx->params.variant == GSEG_FELZ) return level == 0 ? (int)ctx->h_ctl->st.V : GSEG_E_LEVEL;
    if (nl == 0 && level == -1) return (int)ctx->h_ctl->st.V;
    if (level >= nl) return GSEG_E_LEVEL;
    return (int)ctx->h_ctl->stVafter[level];
}

static int level_to_round(const gseg_ctx *ctx, int level, int *round) {
    const int rounds = (int)ctx->h_ctl->st.round;
    if (ctx->params.variant == GSEG_FELZ) {
        if (level != 0 && level != -1) return GSEG_E_LEVEL;
        *round = rounds - 1;
        return GSEG_OK;
    }
    const int nl = (int)ctx->h_ctl->st.levels;
    if (level < 0) level = nl - 1;
    if (level >= nl && !(nl == 0 && level <= 0)) return GSEG_E_LEVEL;
    if (level < 0) level = 0; // no merging round at all (single pixel): round 0's identity map
    *round = level;
    return GSEG_OK;
}

// Label image of the partition after round `round` into dst (device).  Deep hierarchies go through a
// composed table of the late (small) rounds so that a pixel chases 3-4 maps instead of one per round.
// compose_table enqueues the table when the level is deep enough and returns it (else nullptr); a pixel then chases
// the maps of rounds 1..*last and, with a table, looks its label up in it.  k_regions fuses the same chase.
static const u32 *compose_table(gseg_ctx *ctx, int round, int *last) {
    const GsegCtl *h = ctx->h_ctl;
    int first = 1;
    while (first <= round && (h->stV[first] > 65536u || h->map_skip[first])) ++first; // first live round whose input has few components
    if (first >= 1 && first <= round && round - first >= 2 && h->stV[first] <= ctx->Vmax) {
        const u32 n = h->stV[first];
        u32 *F = ctx->d_wsel; // per-round scratch, free once the run is complete
        ++ctx->launches;
        k_compose_table<<<grid_for(n, NT), NT, 0, ctx->stream>>>(ctx->d_ctl, ctx->d_arena, first, round, n, F);
        *last = first - 1;
        return F;
    }
    *last = round;
    return nullptr;
}
template <typename OutT>
static void enqueue_compose(gseg_ctx *ctx, int round, OutT *dst) {
    const size_t V = (size_t)ctx->w * ctx->h;
    int last;
    const u32 *F = compose_table(ctx, round, &last);
    ++ctx->launches;
    if (F) k_compose_px<OutT><<<grid_for(V, NT), NT, 0, ctx->stream>>>(ctx->d_ctl, ctx->d_arena, last + 1, F, dst);
    else k_compose<OutT><<<grid_for(V, NT), NT, 0, ctx->stream>>>(ctx->d_ctl, ctx->d_arena, round, dst);
}

extern "C" int gseg_label_bytes(const gseg_ctx *ctx, int level) {
    const int n = gseg_num_components(ctx, level);
    if (n < 0) return n;
    return n <= 256 ? 1 : (n <= 65536 ? 2 : 4);
}

extern "C" int gseg_labels_ex_async(gseg_ctx *ctx, int level, void *out, int elem_bytes, int mem_kind) {
    if (!ctx || !out || (elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4)) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    if (ctx->graph_mode) return fail(ctx, GSEG_E_STATE, "the last run was an explicit-graph run (no label image)", cudaSuccess);
    int round;
    int rc = level_to_round(ctx, level, &round);
    if (rc) return rc;
    const int need = gseg_label_bytes(ctx, level);
    if (need < 0) return need;
    if (need > elem_bytes) return fail(ctx, GSEG_E_RANGE, "label element type too narrow for this level", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)ctx->w * ctx->h;
    void *dst = mem_kind == GSEG_MEM_DEVICE ? out : (void *)ctx->d_labels[0];
    if (elem_bytes == 4) enqueue_compose<int>(ctx, round, (int *)dst);
    else if (elem_bytes == 2) enqueue_compose<uint16_t>(ctx, round, (uint16_t *)dst);
    else enqueue_compose<uint8_t>(ctx, round, (uint8_t *)dst);
    CK(cudaGetLastError());
    if (mem_kind != GSEG_MEM_DEVICE)
        CK(cudaMemcpyAsync(out, dst, V * (size_t)elem_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return GSEG_OK;
}

extern "C" int gseg_labels_async(gseg_ctx *ctx, int level, int32_t *out, int mem_kind) {
    return gseg_labels_ex_async(ctx, level, out, 4, mem_kind);
}

extern "C" int gseg_labels_ex(gseg_ctx *ctx, int level, void *out, int elem_bytes, int mem_kind) {
    int rc = gseg_labels_ex_async(ctx, level, out, elem_bytes, mem_kind);
    if (rc) return rc;
    return gseg_sync(ctx);
}

// The stored hierarchy: the arena holds one old-id -> new-id map per round back to back, which IS the
// representation the header describes; one linear copy.
extern "C" int gseg_hierarchy_async(gseg_ctx *ctx, uint32_t *out, int64_t cap_entries, int64_t *offsets, int cap_offsets,
                                    int mem_kind) {
    if (!ctx || !offsets) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    if (ctx->graph_mode) return fail(ctx, GSEG_E_STATE, "the last run was an explicit-graph run", cudaSuccess);
    const GsegCtl *h = ctx->h_ctl;
    const size_t V = (size_t)ctx->w * ctx->h;
    if (ctx->params.variant == GSEG_FELZ) { // one level: the final partition
        if (cap_offsets < 2) return GSEG_E_RANGE;
        offsets[0] = 0; offsets[1] = (int64_t)V;
        if (!out) return 1;
        if (cap_entries < (int64_t)V) return GSEG_E_RANGE;
        const int rc = gseg_labels_ex_async(ctx, -1, out, 4, mem_kind);
        return rc ? rc : 1;
    }
    const int nl = (int)h->st.levels > 0 ? (int)h->st.levels : 1; // a run without any merge still has round 0's identity map
    if (cap_offsets < nl + 1) return GSEG_E_RANGE;
    for (int l = 0; l <= nl; ++l) offsets[l] = (int64_t)h->map_off[l];
    if (!out) return nl;
    if (cap_entries < offsets[nl]) return GSEG_E_RANGE;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->d_arena, (size_t)offsets[nl] * sizeof(u32),
                       mem_kind == GSEG_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
    return nl;
}
extern "C" int gseg_hierarchy(gseg_ctx *ctx, uint32_t *out, int64_t cap_entries, int64_t *offsets, int cap_offsets, int mem_kind) {
    const int n = gseg_hierarchy_async(ctx, out, cap_entries, offsets, cap_offsets, mem_kind);
    if (n < 0 || !out) return n;
    const int rc = gseg_sync(ctx);
    return rc ? rc : n;
}

extern "C" int gseg_sync(gseg_ctx *ctx) {
    if (!ctx) return GSEG_E_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

extern "C" int gseg_labels(gseg_ctx *ctx, int level, int32_t *out, int mem_kind) {
    int rc = gseg_labels_async(ctx, level, out, mem_kind);
    if (rc) return rc;
    return gseg_sync(ctx);
}

extern "C" int gseg_labels_all(gseg_ctx *ctx, int32_t *out, int max_levels, int mem_kind) {
    if (!ctx || !out || max_levels < 1) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    int nl = gseg_num_levels(ctx);
    if (nl > max_levels) nl = max_levels;
    const size_t V = (size_t)ctx->w * ctx->h;
    if (ctx->params.variant == GSEG_FELZ) {
        int rc = gseg_labels(ctx, -1, out, mem_kind);
        return rc ? rc : 1;
    }
    if (mem_kind != GSEG_MEM_DEVICE) { int rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64); if (rc) return rc; }
    const int *prev = nullptr;
    for (int l = 0; l < nl; ++l) {
        int *dst = mem_kind == GSEG_MEM_DEVICE ? out + (size_t)l * V : ctx->d_labels[l & 1];
        ++ctx->launches;
        if (l == 0) k_compose<int><<<grid_for(V, NT), NT, 0, ctx->stream>>>(ctx->d_ctl, ctx->d_arena, 0, dst);
        else k_compose_step<<<grid_for(V, NT), NT, 0, ctx->stream>>>(ctx->d_ctl, ctx->d_arena, l, prev, dst);
        if (mem_kind != GSEG_MEM_DEVICE)
            CK(cudaMemcpyAsync(out + (size_t)l * V, dst, V * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        prev = dst;
    }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return nl;
}

extern "C" int gseg_colorize(gseg_ctx *ctx, int level, uint64_t seed, uint8_t *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    int round;
    int rc = level_to_round(ctx, level, &round);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)ctx->w * ctx->h;
    if (mem_kind != GSEG_MEM_DEVICE) rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64); // 4V bytes >= the 3V of the colour image
    if (rc) return rc;
    enqueue_compose<int>(ctx, round, ctx->d_labels[0]);
    uint8_t *dst = mem_kind == GSEG_MEM_DEVICE ? out : (uint8_t *)ctx->d_labels[1];
    ++ctx->launches;
    k_colorize<<<grid_for(V, NT), NT, 0, ctx->stream>>>(ctx->d_labels[0], (u32)V, seed, dst);
    CK(cudaGetLastError());
    if (mem_kind != GSEG_MEM_DEVICE) CK(cudaMemcpyAsync(out, dst, 3 * V, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

// ---- region statistics and pictures (gseg_regions.cuh) ------------------------------------------------------
// Scratch, all of it free once a run is complete: d_wsel (the composed table of deep levels, as gseg_labels_ex),
// d_best[0] (the table on its way to host memory, up to (Vmax + 64) / 8 records; larger ones use d_rtab, allocated by
// GSEG_CAP_REGIONS or on first need), d_labels[1] (host-memory input), d_labels[0] (gseg_render's label image), d_rank
// (mean colours), d_succ (gseg_render's picture on its way to host memory).  d_attr and the edge lists are left alone:
// gseg_export_graph / gseg_strip_record still read them after a run.
static int regions_state(gseg_ctx *ctx, int level, int *round, int *n) {
    if (!ctx->valid) return fail(ctx, GSEG_E_STATE, "no completed segmentation in this context", cudaSuccess);
    if (ctx->graph_mode || ctx->strip_labels)
        return fail(ctx, GSEG_E_STATE, "the last run was an explicit-graph run or a joined strip (no input image)", cudaSuccess);
    int rc = level_to_round(ctx, level, round);
    if (rc) return rc;
    *n = gseg_num_components(ctx, level);
    return *n < 0 ? *n : GSEG_OK;
}

// The image the run read: `rgb` as given (host memory is staged in d_labels[1]), or the context's staged input.
static int regions_input(gseg_ctx *ctx, const uint8_t *rgb, int stride, int kind, const uint8_t **src, long long *sstride) {
    const int w = ctx->w, h = ctx->h;
    if (!rgb) {
        if (!ctx->rgb_staged) return fail(ctx, GSEG_E_STATE, "the run read caller-owned device memory: pass its input", cudaSuccess);
        *src = ctx->d_rgb + (size_t)3 * w * ctx->halo_top;
        *sstride = 3LL * w;
        return GSEG_OK;
    }
    if (stride < 3 * w) return fail(ctx, GSEG_E_ARG, "input stride", cudaSuccess);
    if (kind == GSEG_MEM_DEVICE) { *src = rgb; *sstride = stride; return GSEG_OK; }
    if (kind != GSEG_MEM_HOST) return fail(ctx, GSEG_E_ARG, "rgb_mem_kind", cudaSuccess);
    int rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64); // 4V bytes >= the 3V of the image
    if (rc) return rc;
    uint8_t *d = (uint8_t *)ctx->d_labels[1];
    CK(cudaMemcpy2DAsync(d, (size_t)3 * w, rgb, (size_t)stride, (size_t)3 * w, (size_t)h, cudaMemcpyHostToDevice, ctx->stream));
    *src = d;
    *sstride = 3LL * w;
    return GSEG_OK;
}

// Enqueue the table of the level ending at `round` (n components) into device memory `table`.  Tier: the block-private
// shared-memory table when n <= rg_smem_max and it fits, else global atomics.  Shared-memory fields are 32-bit: a block
// takes at most P = (2^32 - 1) / max(255, w - 1, h - 1) pixels, so no sum of a channel or a coordinate over its pixels
// can exceed 2^32 - 1 (1080p: P = 2.2 M pixels, far above what a block gets anyway).
static int regions_enqueue(gseg_ctx *ctx, int round, u32 n, const uint8_t *src, long long sstride, u64 *table) {
    cudaStream_t s = ctx->stream;
    const u32 w = (u32)ctx->w, h = (u32)ctx->h;
    const u32 cpr = (w + RG_K - 1) / RG_K, nch = cpr * h;
    u32 wide = w - 1 > h - 1 ? w - 1 : h - 1;
    if (wide < 255u) wide = 255u;
    const u64 cpb_max = (0xFFFFFFFFull / wide) / RG_K; // chunks per block that keep the shared fields within 32 bits
    const bool smem = n <= ctx->rg_smem_max && n <= ctx->rg_smem_fit && cpb_max >= 1;
    u64 grid = (u64)ctx->num_sms * 4u;
    const u64 gmax = ((u64)nch + NT - 1) / NT; // at least one chunk per thread
    if (grid > gmax) grid = gmax;
    if (smem && grid < ((u64)nch + cpb_max - 1) / cpb_max) grid = ((u64)nch + cpb_max - 1) / cpb_max;
    if (grid < 1) grid = 1;
    const u32 cpb = (u32)(((u64)nch + grid - 1) / grid);
    grid = ((u64)nch + cpb - 1) / cpb;
    mark_end(ctx, s); // the composed table below is not one of the profiled kernels
    int last;
    const u32 *F = compose_table(ctx, round, &last);
    ctx->rg_n = n;
    mark(ctx, s, "k_regions_init", round);
    k_regions_init<<<grid_for(n, NT), NT, 0, s>>>(table, n);
    if (smem) {
        mark(ctx, s, "k_regions_smem", round);
        k_regions<true><<<(unsigned)grid, NT, (size_t)n * RG_FIELDS * sizeof(u32), s>>>(ctx->d_ctl, ctx->d_arena, last, F, src,
                                                                                        sstride, w, h, n, cpb, table);
    } else {
        mark(ctx, s, "k_regions_gl", round);
        k_regions<false><<<(unsigned)grid, NT, 0, s>>>(ctx->d_ctl, ctx->d_arena, last, F, src, sstride, w, h, n, cpb, table);
    }
    mark_end(ctx, s);
    CK(cudaGetLastError());
    return GSEG_OK;
}

// Device scratch for a table of n records on its way elsewhere.
static int regions_scratch(gseg_ctx *ctx, u32 n, u64 **table) {
    if ((size_t)n * 8 <= ctx->Vmax + 64) { *table = ctx->d_best[0]; return GSEG_OK; }
    int rc = ensure(ctx, &ctx->d_rtab, 8 * (ctx->Vmax + 64));
    *table = ctx->d_rtab;
    return rc;
}

extern "C" int gseg_regions_async(gseg_ctx *ctx, int level, const uint8_t *rgb, int stride, int rgb_mem_kind, uint64_t *out,
                                  int64_t cap_records, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    if (mem_kind == GSEG_MEM_DEVICE && ((uintptr_t)out & 7u)) return fail(ctx, GSEG_E_ARG, "device table not 8-byte aligned", cudaSuccess);
    int round, n;
    int rc = regions_state(ctx, level, &round, &n);
    if (rc) return rc;
    if (cap_records < n) return fail(ctx, GSEG_E_RANGE, "region table capacity below the component count", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    const uint8_t *src;
    long long sstride;
    rc = regions_input(ctx, rgb, stride, rgb_mem_kind, &src, &sstride);
    if (rc) return rc;
    u64 *table = (u64 *)out;
    if (mem_kind != GSEG_MEM_DEVICE && (rc = regions_scratch(ctx, (u32)n, &table)) != 0) return rc;
    rc = regions_enqueue(ctx, round, (u32)n, src, sstride, table);
    if (rc) return rc;
    if (mem_kind != GSEG_MEM_DEVICE) CK(cudaMemcpyAsync(out, table, (size_t)n * 64, cudaMemcpyDeviceToHost, ctx->stream));
    return n;
}

extern "C" int gseg_regions(gseg_ctx *ctx, int level, const uint8_t *rgb, int stride, int rgb_mem_kind, uint64_t *out,
                            int64_t cap_records, int mem_kind) {
    const int n = gseg_regions_async(ctx, level, rgb, stride, rgb_mem_kind, out, cap_records, mem_kind);
    if (n < 0) return n;
    const int rc = gseg_sync(ctx);
    return rc ? rc : n;
}

extern "C" int gseg_render(gseg_ctx *ctx, int level, int mode, uint32_t colour, const uint8_t *rgb, int stride, int rgb_mem_kind,
                           uint8_t *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (mode != GSEG_RENDER_MEAN && mode != GSEG_RENDER_OVERLAY && mode != GSEG_RENDER_BOUNDARY) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    int round, n;
    int rc = regions_state(ctx, level, &round, &n);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const u32 w = (u32)ctx->w, h = (u32)ctx->h;
    const size_t V = (size_t)w * h;
    const uint8_t *src = nullptr;
    long long sstride = 0;
    if (mode != GSEG_RENDER_BOUNDARY && (rc = regions_input(ctx, rgb, stride, rgb_mem_kind, &src, &sstride)) != 0) return rc;
    const u32 *mean = nullptr;
    if (mode == GSEG_RENDER_MEAN) {
        u64 *table;
        if ((rc = regions_scratch(ctx, (u32)n, &table)) != 0) return rc;
        if ((rc = regions_enqueue(ctx, round, (u32)n, src, sstride, table)) != 0) return rc;
        mark(ctx, s, "k_region_means", round);
        k_region_means<<<grid_for((size_t)n, NT), NT, 0, s>>>(table, (u32)n, ctx->d_rank);
        mean = ctx->d_rank;
    }
    mark_end(ctx, s);
    enqueue_compose<int>(ctx, round, ctx->d_labels[0]);
    uint8_t *dst = mem_kind == GSEG_MEM_DEVICE ? out : (uint8_t *)ctx->d_succ; // 4V bytes >= the 3V of a picture
    const int aligned = ((uintptr_t)dst & 3u) == 0;
    const int g = grid_for((V + 3) / 4, NT);
    if (mode == GSEG_RENDER_MEAN) {
        mark(ctx, s, "k_render_mean", round);
        k_render<GSEG_RENDER_MEAN_><<<g, NT, 0, s>>>(ctx->d_labels[0], w, h, mean, src, sstride, colour, dst, aligned);
    } else if (mode == GSEG_RENDER_OVERLAY) {
        mark(ctx, s, "k_render_overlay", round);
        k_render<GSEG_RENDER_OVERLAY_><<<g, NT, 0, s>>>(ctx->d_labels[0], w, h, mean, src, sstride, colour, dst, aligned);
    } else {
        mark(ctx, s, "k_render_boundary", round);
        k_render<GSEG_RENDER_BOUNDARY_><<<g, NT, 0, s>>>(ctx->d_labels[0], w, h, mean, src, sstride, colour, dst, aligned);
    }
    mark_end(ctx, s);
    CK(cudaGetLastError());
    if (mem_kind != GSEG_MEM_DEVICE)
        CK(cudaMemcpyAsync(out, dst, V * (mode == GSEG_RENDER_BOUNDARY ? 1 : 3), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return GSEG_OK;
}

extern "C" int gseg_weights(gseg_ctx *ctx, float *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)ctx->w * ctx->h, n = V * ctx->D;
    CK(cudaMemcpyAsync(out, ctx->d_wgrid, n * sizeof(float),
                       mem_kind == GSEG_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

extern "C" int gseg_blurred(gseg_ctx *ctx, float *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)ctx->w * ctx->h;
    CK(cudaMemcpyAsync(out, ctx->d_planes, 3 * V * sizeof(float),
                       mem_kind == GSEG_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

// ---- tiled schedule: export / import of component graphs ------------------------------------------------
// Device side of the export: gather the pages into a dense list and, if asked, eliminate duplicates.
// Leaves the list in (x_ab, x_w) with x_count entries and caches it until the next run.
static int export_prepare(gseg_ctx *ctx, int dedup) {
    if (ctx->x_valid && ctx->x_dedup == (dedup != 0)) return GSEG_OK;
    const GsegCtl *h = ctx->h_ctl;
    const size_t V = h->st.V, E = h->st.E;
    const int cur = (int)(h->st.round & 1u);
    const GsegBufs B = bufs_of(ctx);
    const u32 P = h->st.P;
    cudaStream_t s = ctx->stream;
    if (P) {
        ctx->launches += 2;
        k_export_scan<<<1, 1024, 0, s>>>(B, cur, P);
        k_export_gather<<<grid_for(P, NT / 32), NT, 0, s>>>(B, cur, P);
        CK(cudaGetLastError());
    }
    ctx->x_ab = ctx->d_eab[cur ^ 1]; ctx->x_w = ctx->d_ew[cur ^ 1]; ctx->x_count = E;
    if (dedup && E > 1) {
        if (ctx->x_cap < E) return fail(ctx, GSEG_E_SIZE, "graph export with duplicate elimination: more live edges than the context's de-duplication arrays hold", cudaSuccess);
        int bits = 1;
        while (bits < 64 && ((u64)V * V - 1u) >> bits) ++bits; // pair keys are < V^2
        ctx->launches += 3;
        k_pair_keys<<<grid_for(E, NT), NT, 0, s>>>(ctx->x_ab, (u32)E, (u32)V, ctx->d_xkeys, ctx->d_xvals, ctx->d_xkeep);
        CK(cudaGetLastError());
        cudaError_t e = onesweep_sort_pairs(&ctx->sort, ctx->d_xkeys, ctx->d_xvals, E, 0, bits, s);
        if (e != cudaSuccess) return fail(ctx, GSEG_E_CUDA, "onesweep_sort_pairs", e);
        // minimum (weight, list position) of every run of equal pairs, in parallel (segmented warp minima + one atomic per
        // run part), then the winners' flags
        CK(cudaMemsetAsync(ctx->d_winner, 0xFF, E * sizeof(u64), s));
        k_pair_select_runs<<<grid_for(E, NT), NT, 0, s>>>(ctx->d_xkeys, ctx->d_xvals, ctx->x_w, (u32)E, ctx->d_winner);
        k_pair_mark_runs<<<grid_for(E, NT), NT, 0, s>>>(ctx->d_xkeys, ctx->d_winner, (u32)E, ctx->d_xkeep);
        ++ctx->launches;
        CK(cudaMemsetAsync(&ctx->d_ctl->ticketE, 0, sizeof(u32), s));
        const u32 tag = ctx->epoch_next; // a tag no round of any run uses
        ctx->epoch_next += 2u;
        k_compact_keep<<<grid_for(E, 1024, 64), 1024, 0, s>>>(ctx->d_ctl, ctx->x_ab, ctx->x_w, ctx->d_xkeep, (u32)E, tag,
                                                                ctx->d_statusE, ctx->d_xab, ctx->d_xw);
        CK(cudaGetLastError());
        u32 kept = 0;
        CK(cudaMemcpyAsync(&kept, &ctx->d_ctl->Eacc[GSEG_MAXR], sizeof(u32), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        ctx->x_ab = ctx->d_xab; ctx->x_w = ctx->d_xw; ctx->x_count = kept;
    }
    ctx->x_valid = true; ctx->x_dedup = dedup != 0;
    return GSEG_OK;
}

extern "C" int gseg_export_graph(gseg_ctx *ctx, int dedup, int64_t *n_components, int64_t *n_edges, uint32_t *size, float *Int,
                                 uint32_t *ea, uint32_t *eb, float *w, int64_t cap_components, int64_t cap_edges) {
    if (!ctx || !n_components || !n_edges) return GSEG_E_ARG;
    if (!ctx->valid || ctx->params.variant == GSEG_SUPERPIX) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    int rc = export_prepare(ctx, dedup);
    if (rc) return rc;
    const GsegCtl *h = ctx->h_ctl;
    const int64_t V = h->st.V, E = (int64_t)ctx->x_count;
    *n_components = V; *n_edges = E;
    if (!size && !Int && !ea && !eb && !w) return GSEG_OK;
    if (!size || !Int || !ea || !eb || !w || cap_components < V || cap_edges < E) return GSEG_E_ARG;
    const int cur = (int)(h->st.round & 1u);
    std::vector<uint2> hab, hat;
    try { hab.resize((size_t)E); hat.resize((size_t)V); } catch (...) { return fail(ctx, GSEG_E_ARG, "host staging allocation", cudaSuccess); }
    if (E) {
        CK(cudaMemcpyAsync(hab.data(), ctx->x_ab, (size_t)E * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaMemcpyAsync(w, ctx->x_w, (size_t)E * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaMemcpyAsync(hat.data(), ctx->d_attr[cur], (size_t)V * sizeof(uint2), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int64_t i = 0; i < E; ++i) { ea[i] = hab[(size_t)i].x; eb[i] = hab[(size_t)i].y; }
    for (int64_t i = 0; i < V; ++i) { size[i] = hat[(size_t)i].x; memcpy(&Int[i], &hat[(size_t)i].y, 4); }
    return GSEG_OK;
}

extern "C" int gseg_blurred_rows(gseg_ctx *ctx, int y0, int nrows, float *out, int mem_kind) {
    if (!ctx || !out) return GSEG_E_ARG;
    if (!ctx->valid) return GSEG_E_STATE;
    if (y0 < 0 || nrows < 1 || y0 + nrows > ctx->h) return GSEG_E_ARG;
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)ctx->w * ctx->h, n = (size_t)nrows * ctx->w;
    for (int c = 0; c < 3; ++c) // one linear copy per plane (a pitched copy's pitch would be V * 4 bytes: beyond CUDA's limit for large strips)
        CK(cudaMemcpyAsync(out + (size_t)c * n, ctx->d_planes + (size_t)c * V + (size_t)y0 * ctx->w, n * sizeof(float),
                           mem_kind == GSEG_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

static int wait_rounds(gseg_ctx *ctx);

// The Boruvka rounds on an explicit graph that already sits in the context's buffers: attr[1][0..V), eab[1] /
// ew[1][0..E) in list order, best[1][0..V) = none.  Leaves the composed label of every input component in
// d_wsel and returns the number of final components (or a negative status).
static int graph_run(gseg_ctx *ctx, size_t V, size_t E, const gseg_params *p) {
    cudaStream_t s = ctx->stream;
    ctx->valid = false; ctx->x_valid = false; ctx->graph_mode = true;
    ctx->params = *p;
    ctx->w = (int)V; ctx->h = 1; ctx->D = 2;
    const int R = max_rounds_of(p);
    if (ctx->epoch_next + GSEG_EPOCHS_PER_RUN >= (1u << 30)) {
        CK(cudaMemsetAsync(ctx->d_statusC, 0, ctx->ntilesC * sizeof(u64), s));
        CK(cudaMemsetAsync(ctx->d_statusE, 0, ctx->ntilesE * sizeof(u64), s));
        ctx->epoch_next = 1;
    }
    GsegHead *hh = ctx->h_head;
    GsegRunParams *hp = &hh->p;
    memset(hp, 0, sizeof(*hp));
    hp->w = (int)V; hp->h = 1; hp->h_in = 1; hp->D = 2; hp->variant = p->variant;
    hp->k = p->k; hp->min_size = p->min_size; hp->max_rounds = R + 1 > GSEG_MAXR ? GSEG_MAXR : R + 1; // rounds are numbered from 1 here
    hp->max_levels = p->max_levels > 0 ? p->max_levels : INT_MAX;
    hp->arena_cap = (u32)ctx->arena_cap; hp->edge_slots = (u32)edge_slots(ctx);
    hp->epoch_base = ctx->epoch_next;
    hp->filter_shift = ctx->filter_shift;
    const bool host_loop = (p->flags & GSEG_FLAG_HOST_LOOP) != 0;
    hp->tail_E = ctx->run_tail_E = host_loop ? 0u : ctx->tail_E;
    hp->tail_V = ctx->run_tail_V = host_loop ? 0u : ctx->tail_V;
    hp->tail_P = ctx->tail_P;
    hp->no_dedup = dedup_enabled(ctx) ? 0u : 1u; hp->dd_V = dedup_V(ctx);
    ctx->epoch_next += GSEG_EPOCHS_PER_RUN;
    const u32 P = (u32)((E + GSEG_PAGE - 1) / GSEG_PAGE);
    hh->st.V = (u32)V; hh->st.E = (u32)E; hh->st.round = 1; hh->st.phase = PH_PRED; hh->st.levels = 0; hh->st.map_off = 0;
    hh->st.P = P; hh->st.pad = 0;
    hh->Vnext = (u32)V; hh->error = DERR_NONE; hh->ticketC = 0; hh->ticketE = 0; hh->doneE = 0;
    memset(hh->Eacc, 0, sizeof(hh->Eacc));
    memset(hh->map_skip, 0, sizeof(hh->map_skip)); hh->resume_phase = PH_DONE;
    memset(hh->stDedupIn, 0, sizeof(hh->stDedupIn)); memset(hh->stDedupOut, 0, sizeof(hh->stDedupOut));
    CK(cudaMemcpyAsync(ctx->d_ctl, hh, sizeof(GsegHead), cudaMemcpyHostToDevice, s));
    ctx->n_marks = 0;
    const GsegBufs B = bufs_of(ctx);
    if (P) { ++ctx->launches; k_graph_init<<<grid_for(P, NT / 32), NT, 0, s>>>(B, (u32)E, P); }
    CK(cudaGetLastError());
    // the usual schedule from round 1 on; a joined graph is small, so normally everything runs in the tail
    ctx->nbig_hint = -1;
    int rc;
    if (host_loop) {
        rc = readback(ctx);
        for (int go; !rc && (go = run_continues(ctx)) != 0;) {
            if (go < 0) { rc = go; break; }
            if (dedup_wanted_host(ctx)) {
                enqueue_dedup(ctx, s, (int)ctx->h_ctl->st.round);
                CK(cudaGetLastError());
                if ((rc = readback(ctx)) != 0) break;
            }
            enqueue_round(ctx, s, (int)ctx->h_ctl->st.round, ctx->h_ctl->st.V, ctx->h_ctl->st.P);
            CK(cudaGetLastError());
            rc = readback(ctx);
        }
    } else {
        if (dedup_enabled(ctx)) enqueue_dedup(ctx, s, -1);
        CK(cudaGetLastError());
        CK(enqueue_tail(ctx, s));
        ctx->pending = true;
        rc = wait_rounds(ctx);
    }
    ctx->pending = false;
    if (rc) return rc;
    if (ctx->h_ctl->error == DERR_SCAN) return fail(ctx, GSEG_E_INTERNAL, "look-back watchdog", cudaSuccess);
    if (ctx->h_ctl->error == DERR_ARENA) return fail(ctx, GSEG_E_ARENA, "map arena", cudaSuccess);
    if (ctx->h_ctl->error == DERR_CHASE) return fail(ctx, GSEG_E_INTERNAL, "successor cycle", cudaSuccess);
    if (ctx->h_ctl->error >= DERR_CHECK) {
        snprintf(ctx->err, sizeof(ctx->err), "checked build: bounds check at site %u failed", ctx->h_ctl->error - DERR_CHECK);
        return GSEG_E_INTERNAL;
    }
    // labels of the input components: the maps of rounds 1 .. last composed
    const int last = (int)ctx->h_ctl->st.round - 1;
    ++ctx->launches;
    k_compose_table<<<grid_for(V, NT), NT, 0, s>>>(ctx->d_ctl, ctx->d_arena, 1, last, (u32)V, ctx->d_wsel);
    CK(cudaGetLastError());
    return (int)ctx->h_ctl->st.V;
}


extern "C" int gseg_segment_graph(gseg_ctx *ctx, int64_t n_components, const uint32_t *size, const float *Int, int64_t n_edges,
                                  const uint32_t *ea, const uint32_t *eb, const float *w, const gseg_params *p,
                                  int32_t *labels_out) {
    if (!ctx || !p || !labels_out || n_components < 1 || n_edges < 0 || !size || !Int || (n_edges && (!ea || !eb || !w)))
        return GSEG_E_ARG;
    if (ctx->pending) return fail(ctx, GSEG_E_STATE, "previous run not waited for", cudaSuccess);
    if (p->variant != GSEG_FELZ && p->variant != GSEG_HIER) return fail(ctx, GSEG_E_ARG, "graph rounds: FELZ or HIER", cudaSuccess);
    if (!(p->k >= 0.0f) || p->min_size < 0 || p->max_rounds < 0 || p->max_levels < 0) return fail(ctx, GSEG_E_ARG, "parameter range", cudaSuccess);
    if ((size_t)n_components > ctx->Vmax || (size_t)n_edges + GSEG_PAGE > edge_slots(ctx))
        return fail(ctx, GSEG_E_SIZE, "graph exceeds context capacity", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)n_components, E = (size_t)n_edges;
    std::vector<uint2> hab, hat;
    try { hab.resize(E); hat.resize(V); } catch (...) { return fail(ctx, GSEG_E_ARG, "host staging allocation", cudaSuccess); }
    // every comparison of the engine orders fp32 values by their bit patterns: only non-negative, non-NaN
    // weights and Int(C) order like their values (-0.0 would sort above every finite weight)
    auto bad_float = [](float f) { u32 b; memcpy(&b, &f, 4); return (b >> 31) != 0u || b > GSEG_INF_BITS; };
    for (size_t i = 0; i < E; ++i) {
        if (ea[i] >= V || eb[i] >= V || ea[i] == eb[i]) return fail(ctx, GSEG_E_ARG, "edge end out of range or self-loop", cudaSuccess);
        if (bad_float(w[i])) return fail(ctx, GSEG_E_ARG, "edge weight negative (sign bit set) or NaN", cudaSuccess);
        hab[i] = make_uint2(ea[i], eb[i]);
    }
    for (size_t i = 0; i < V; ++i) {
        if (bad_float(Int[i])) return fail(ctx, GSEG_E_ARG, "Int(C) negative (sign bit set) or NaN", cudaSuccess);
        hat[i].x = size[i]; memcpy(&hat[i].y, &Int[i], 4);
    }
    cudaStream_t s = ctx->stream;
    if (E) {
        CK(cudaMemcpyAsync(ctx->d_eab[1], hab.data(), E * sizeof(uint2), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(ctx->d_ew[1], w, E * sizeof(u32), cudaMemcpyHostToDevice, s));
    }
    CK(cudaMemcpyAsync(ctx->d_attr[1], hat.data(), V * sizeof(uint2), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(ctx->d_best[1], 0xFF, V * sizeof(u64), s));
    CK(cudaStreamSynchronize(s)); // the staging vectors die with this scope
    const int n = graph_run(ctx, V, E, p);
    if (n < 0) return n;
    CK(cudaMemcpyAsync(labels_out, ctx->d_wsel, V * sizeof(u32), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return n;
}

// ---- tiled schedule on the device: strip record, join, joined rounds ----------------------------------------
extern "C" int gseg_strip_record(gseg_ctx *ctx, int dedup, void *dev_out, int64_t cap_bytes, int64_t *bytes) {
    if (!ctx || !bytes) return GSEG_E_ARG;
    if (!ctx->valid || ctx->graph_mode || ctx->params.variant == GSEG_SUPERPIX) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    int rc = export_prepare(ctx, dedup);
    if (rc) return rc;
    const GsegCtl *h = ctx->h_ctl;
    const size_t nV = h->st.V, nE = ctx->x_count, w = (size_t)ctx->w;
    *bytes = (int64_t)(rec_words(nV, nE, w) * sizeof(u32));
    if (!dev_out) return GSEG_OK;
    if (cap_bytes < *bytes) return GSEG_E_RANGE;
    cudaStream_t s = ctx->stream;
    u32 *rec = (u32 *)dev_out;
    const int cur = (int)(h->st.round & 1u);
    // the strip's dense label image stays in d_labels[0]: gseg_join_segment maps it through the joined result
    int round;
    rc = level_to_round(ctx, -1, &round);
    if (rc) return rc;
    enqueue_compose<int>(ctx, round, ctx->d_labels[0]);
    CK(cudaMemcpyAsync(rec + GSEG_REC_HEAD, ctx->d_attr[cur], nV * sizeof(uint2), cudaMemcpyDeviceToDevice, s));
    if (nE) {
        CK(cudaMemcpyAsync(rec + GSEG_REC_HEAD + 2 * nV, ctx->x_ab, nE * sizeof(uint2), cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(rec + GSEG_REC_HEAD + 2 * nV + 2 * nE, ctx->x_w, nE * sizeof(u32), cudaMemcpyDeviceToDevice, s));
    }
    ++ctx->launches;
    k_record_rows<<<grid_for(w, NT), NT, 0, s>>>(ctx->d_labels[0], ctx->d_planes, (u32)ctx->w, (u32)ctx->h, (u32)nV, (u32)nE, rec);
    CK(cudaGetLastError());
    ctx->strip_w = ctx->w; ctx->strip_h = ctx->h; ctx->strip_nV = (u32)nV; ctx->strip_labels = true;
    CK(cudaStreamSynchronize(s));
    return GSEG_OK;
}

extern "C" int gseg_join_segment(gseg_ctx *ctx, const void *dev_records, int n_strips, int64_t record_stride_bytes, int my_strip,
                                 const gseg_params *p, void *labels_out, int elem_bytes, int mem_kind, int64_t *n_joined_components,
                                 int64_t *n_joined_edges) {
    if (!ctx || !dev_records || !p || n_strips < 1 || n_strips > GSEG_MAX_STRIPS || my_strip < 0 || my_strip >= n_strips ||
        record_stride_bytes < (int64_t)(GSEG_REC_HEAD * sizeof(u32)) || (record_stride_bytes & 3))
        return GSEG_E_ARG;
    if (labels_out && elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    if (ctx->pending) return fail(ctx, GSEG_E_STATE, "previous run not waited for", cudaSuccess);
    if (!ctx->strip_labels) return fail(ctx, GSEG_E_STATE, "gseg_strip_record has not been called for this strip", cudaSuccess);
    if (p->variant != GSEG_FELZ && p->variant != GSEG_HIER) return fail(ctx, GSEG_E_ARG, "graph rounds: FELZ or HIER", cudaSuccess);
    if (p->connectivity != 4 && p->connectivity != 8) return fail(ctx, GSEG_E_ARG, "connectivity must be 4 or 8", cudaSuccess);
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    // the record headers (32 bytes each) are the only thing the host reads
    u32 heads[GSEG_MAX_STRIPS][GSEG_REC_HEAD];
    CK(cudaMemcpy2DAsync(heads, sizeof(heads[0]), dev_records, (size_t)record_stride_bytes, sizeof(heads[0]), (size_t)n_strips,
                         cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    JoinDesc jd;
    memset(&jd, 0, sizeof(jd));
    jd.n_strips = (u32)n_strips; jd.w = heads[0][3]; jd.conn = (u32)p->connectivity;
    jd.ncut = p->connectivity == 8 ? jd.w + 2u * (jd.w - 1u) : jd.w;
    jd.stride_words = (unsigned long long)record_stride_bytes / 4u;
    u64 vo = 0, eo = 0;
    for (int i = 0; i < n_strips; ++i) {
        if (heads[i][0] != GSEG_REC_MAGIC || heads[i][3] != jd.w) return fail(ctx, GSEG_E_ARG, "not a strip record (or strips of different widths)", cudaSuccess);
        if ((u64)rec_words(heads[i][1], heads[i][2], jd.w) * 4u > (u64)record_stride_bytes) return fail(ctx, GSEG_E_ARG, "record stride shorter than a record", cudaSuccess);
        jd.voff[i] = (u32)vo; jd.eoff[i] = (u32)eo; jd.ne[i] = heads[i][2];
        vo += heads[i][1];
        eo += heads[i][2] + (i + 1 < n_strips ? jd.ncut : 0u);
    }
    jd.voff[n_strips] = (u32)vo; jd.eoff[n_strips] = (u32)eo;
    if (vo > ctx->Vmax || eo + GSEG_PAGE > edge_slots(ctx) || vo >= 0xFFFFFFFFull || eo >= 0xFFFFFFFFull)
        return fail(ctx, GSEG_E_SIZE, "joined graph exceeds context capacity", cudaSuccess);
    if ((u32)ctx->strip_w != jd.w || heads[my_strip][1] != ctx->strip_nV) return fail(ctx, GSEG_E_ARG, "my_strip is not this context's record", cudaSuccess);
    if (n_joined_components) *n_joined_components = (int64_t)vo;
    if (n_joined_edges) *n_joined_edges = (int64_t)eo;
    ++ctx->launches;
    k_join<<<grid_for(vo + eo, NT), NT, 0, s>>>(jd, (const u32 *)dev_records, bufs_of(ctx));
    CK(cudaGetLastError());
    const int n = graph_run(ctx, (size_t)vo, (size_t)eo, p);
    if (n < 0) return n;
    if (labels_out) {
        const size_t Vs = (size_t)ctx->strip_w * ctx->strip_h;
        void *dst = labels_out;
        if (mem_kind != GSEG_MEM_DEVICE) { int rc = ensure(ctx, &ctx->d_labels[1], ctx->Vmax + 64); if (rc) return rc; dst = ctx->d_labels[1]; }
        if (elem_bytes == 1 ? n > 256 : (elem_bytes == 2 ? n > 65536 : false)) return fail(ctx, GSEG_E_RANGE, "label element type too narrow", cudaSuccess);
        ++ctx->launches;
        const int g = grid_for(Vs, NT);
        if (elem_bytes == 4) k_map_labels<int><<<g, NT, 0, s>>>(ctx->d_labels[0], ctx->d_wsel, jd.voff[my_strip], Vs, (int *)dst);
        else if (elem_bytes == 2) k_map_labels<uint16_t><<<g, NT, 0, s>>>(ctx->d_labels[0], ctx->d_wsel, jd.voff[my_strip], Vs, (uint16_t *)dst);
        else k_map_labels<uint8_t><<<g, NT, 0, s>>>(ctx->d_labels[0], ctx->d_wsel, jd.voff[my_strip], Vs, (uint8_t *)dst);
        CK(cudaGetLastError());
        if (mem_kind != GSEG_MEM_DEVICE) CK(cudaMemcpyAsync(labels_out, dst, Vs * (size_t)elem_bytes, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    return n;
}

extern "C" int gseg_stats(const gseg_ctx *ctx, gseg_round_stat *out, int cap) {
    if (!ctx || !ctx->valid) return GSEG_E_STATE;
    const GsegCtl *hc = ctx->h_ctl;
    const int n = (int)hc->st.round;
    bool deduped = false; // the list entering round i has had duplicates removed (by the sort step in front of it or of an earlier round)
    for (int i = 0; i < n && i < cap && out; ++i) {
        if (hc->stDedupOut[i]) deduped = true;
        out[i].n_components = hc->stV[i];
        // the sort step knows both counts of the round it ran in front of; n_edges stays the list as it was carried
        out[i].n_edges = i == 0 ? 0 : (hc->stDedupIn[i] ? hc->stDedupIn[i] : hc->stE[i]);
        out[i].n_merged = hc->stM[i];
        out[i].phase = (int32_t)hc->stP[i];
        const bool tail = hc->stTail[i] != 0;
        out[i].in_tail = tail ? 1 : 0;
        out[i].n_pages = (int32_t)hc->stPages[i];
        out[i].n_edges_dedup = deduped ? (int32_t)(hc->stDedupOut[i] ? hc->stDedupOut[i] : hc->stE[i]) : 0;
        out[i].us_end = (float)((double)(hc->t_end[i] - hc->t_start) * 1e-3);
        out[i].us_S = tail ? (float)((double)(hc->t_S[i] - hc->t_begin[i]) * 1e-3) : 0.f;
        out[i].us_R = tail ? (float)((double)(hc->t_R[i] - hc->t_S[i]) * 1e-3) : 0.f;
        out[i].us_E = tail ? (float)((double)(hc->t_end[i] - hc->t_R[i]) * 1e-3) : 0.f;
    }
    return n;
}

extern "C" int gseg_synth_rows(gseg_ctx *ctx, uint8_t *out, int w, int y_first, int nrows, uint64_t seed, int mem_kind) {
    if (!ctx || !out || w < 1 || nrows < 1 || y_first < 0) return GSEG_E_ARG;
    if (mem_kind != GSEG_MEM_HOST && mem_kind != GSEG_MEM_DEVICE) return GSEG_E_ARG;
    if (mem_kind == GSEG_MEM_HOST && (size_t)w * nrows > ctx->Vmax) return GSEG_E_SIZE; // staged through the context
    if (ctx->pending) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    const size_t V = (size_t)w * nrows;
    uint8_t *dst = mem_kind == GSEG_MEM_DEVICE ? out : ctx->d_rgb;
    ++ctx->launches;
    k_synth<<<grid_for(V, NT), NT, 0, ctx->stream>>>(dst, w, nrows, seed, y_first);
    CK(cudaGetLastError());
    if (mem_kind != GSEG_MEM_DEVICE) CK(cudaMemcpyAsync(out, dst, 3 * V, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return GSEG_OK;
}

extern "C" int gseg_synth(gseg_ctx *ctx, uint8_t *out, int w, int h, uint64_t seed, int mem_kind) {
    return gseg_synth_rows(ctx, out, w, 0, h, seed, mem_kind);
}

extern "C" int gseg_sort_pairs_u64(gseg_ctx *ctx, uint64_t *keys, uint32_t *vals, int64_t n, int begin_bit, int end_bit) {
    if (!ctx || !keys || n < 0 || begin_bit < 0 || end_bit > 64 || begin_bit >= end_bit) return GSEG_E_ARG;
    CK(cudaSetDevice(ctx->device));
    // The scratch is reallocated exactly when a capacity grows.  Its addresses are no test: a buffer freed and allocated
    // again can come back at the same address while another one moved.
    const size_t cap_n = ctx->sort.cap_n, cap_status = ctx->sort.cap_status;
    cudaError_t e = onesweep_sort_pairs(&ctx->sort, (u64 *)keys, (u32 *)vals, (size_t)n, begin_bit, end_bit, ctx->stream);
    if (e != cudaSuccess) return fail(ctx, GSEG_E_CUDA, "onesweep_sort_pairs", e);
    CK(cudaStreamSynchronize(ctx->stream));
    if (cap_n != ctx->sort.cap_n || cap_status != ctx->sort.cap_status) CK(upload_dd(ctx)); // a larger sort than any before: the scratch moved
    return GSEG_OK;
}

// ---- profiling / accounting ----------------------------------------------------------------------
extern "C" int gseg_set_profiling(gseg_ctx *ctx, int on) {
    if (!ctx) return GSEG_E_ARG;
    ctx->profiling = on != 0;
    ctx->n_marks = 0;
    return GSEG_OK;
}

extern "C" long long gseg_launch_count(const gseg_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" long long gseg_compaction_count(const gseg_ctx *ctx) { return ctx ? ctx->compactions : 0; }

// Algorithmic bytes of one kernel launch, SURVEY.md section 8(d) accounting: every input array read once, every
// output written once, gathers at element size, and the per-component minimum as ONE 8-byte word per component
// of the next round (section 8(d) "min-edge select: 8 V write"), not 8 bytes per atomic.  strict = the same with
// every gathered array counted once however many elements gather from it.  E0 = grid edges that exist.
static void algo_bytes(const gseg_ctx *c, const char *name, int r, double *algo, double *strict) {
    const GsegCtl *h = c->h_ctl;
    *algo = *strict = 0;
    if (r < 0) return;
    const double W = c->w, H = c->h, V0 = W * H;
    const double E0 = c->D == 2 ? 2 * V0 - W - H : 4 * V0 - 3 * W - 3 * H + 2;
    const double V = r == 0 ? V0 : h->stV[r], E = r == 0 ? 0 : h->stE[r], Vn = h->stVafter[r];
    const double En = (r + 1 < (int)h->st.round) ? h->stE[r + 1] : h->st.E;
    const bool sp = c->params.variant == GSEG_SUPERPIX;
    const double acc = sp ? 40 : 16; // cleared accumulators per new component: (size, Int) 8 + minimum 8 [+ 3 colour sums 24]
    double a = 0, s = 0;
    if (!strcmp(name, "k_blur_tile") || !strcmp(name, "k_blur_h")) a = s = 3 * V0 + 12 * V0;   // u8 image in, 3 fp32 planes out
    else if (!strcmp(name, "k_blur_v")) a = s = 12 * V0 + 12 * V0;
    else if (!strcmp(name, "k_sobel")) a = s = 12 * V0 + 4 * V0;
    // planes (+G) in; weights out (4 E0), successor + chosen weight out (8 V), new id of every root + its cleared accumulators
    else if (!strcmp(name, "k_r0_graph")) a = s = (sp ? 16 : 12) * V0 + 4 * E0 + 8 * V0 + (4 + acc) * Vn;
    // pointer jump (one pass): succ in, one 4-byte gather up the chain; new id of the root: a 4-byte gather; map out;
    // contraction: old (size, Int) [+ colour sums] in, chosen weight of the merged in, (size, Int) [+ sums] per new component out
    else if (!strcmp(name, "k_relabel")) {
        const double attr_in = r == 0 ? (sp ? 12 * V : 0) : (sp ? 32 : 8) * V, out = (sp ? 32 : 8) * Vn;
        a = 4 * V + 4 * V + 4 * V + 4 * V + attr_in + 4 * (V - Vn) + out;
        s = 4 * V + 4 * Vn + 4 * V + attr_in + 4 * (V - Vn) + out; // the chain is inside succ[], the ids gathered are Vn distinct words
    }
    // grid edges: weight in (the ends are implicit), both ends' new ids gathered (4 + 4), survivors out (12), one minimum per component
    else if (!strcmp(name, "k_r0_edges") || !strcmp(name, "k_r0_edges_rl")) { a = 4 * E0 + 8 * E0 + 12 * En + 8 * Vn; s = 4 * E0 + 4 * V0 + 12 * En + 8 * Vn; }
    // per component: its minimum in (8), that edge's ends gathered (8), (size, Int) of both ends (16) and the partner's
    // minimum (8) gathered; successor + chosen weight out (8); new id of every root + its cleared accumulators
    else if (!strcmp(name, "k_succ_scan")) { a = 8 * V + 8 * V + 16 * V + 8 * V + 8 * V + (4 + acc) * Vn; s = 8 * V + 8 * V + 8 * V + 8 * V + (4 + acc) * Vn; }
    // 12 B per edge in, both ends' new ids gathered, 12 B per survivor out, one minimum per component
    // (superpixel: + both ends' 16-byte means gathered per survivor)
    else if (!strcmp(name, "k_edges")) { a = 12 * E + 8 * E + 12 * En + 8 * Vn + (sp ? 32 * En : 0); s = 12 * E + 4 * V + 12 * En + 8 * Vn + (sp ? 16 * Vn : 0); }
    else if (!strcmp(name, "k_means")) a = s = 32 * Vn + 16 * Vn;
    else if (!strcmp(name, "k_page_scan")) a = s = 8.0 * h->stPages[r];
    // region statistics (gseg_regions.cuh): the input (3 V) and the round-0 map of the fused label chase (4 V) in, the
    // table (64 B per component) out; later maps and the composed table are gathers of few components (cached)
    else if (!strcmp(name, "k_regions_smem") || !strcmp(name, "k_regions_gl")) a = s = 3 * V0 + 4 * V0 + 64.0 * c->rg_n;
    else if (!strcmp(name, "k_regions_init")) a = s = 64.0 * c->rg_n;
    else if (!strcmp(name, "k_region_means")) a = s = 32.0 * c->rg_n + 4.0 * c->rg_n;
    // pictures: the label image in (4 V; the stencil's neighbours are the same array), the picture out
    else if (!strcmp(name, "k_render_mean")) { a = 4 * V0 + 4 * V0 + 3 * V0; s = 4 * V0 + 4.0 * c->rg_n + 3 * V0; }
    else if (!strcmp(name, "k_render_overlay")) a = s = 4 * V0 + 3 * V0 + 3 * V0;
    else if (!strcmp(name, "k_render_boundary")) a = s = 4 * V0 + V0;
    *algo = a; *strict = s;
}

extern "C" int gseg_profile_read(gseg_ctx *ctx, gseg_kernel_time *out, int cap) {
    if (!ctx || !ctx->valid) return GSEG_E_STATE;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    int n = 0;
    for (int i = 0; i + 1 < ctx->n_marks && n < cap; ++i) {
        // the closing event of mark i is the next mark's event; nameless marks are read-back gaps
        if (!ctx->mark_name[i]) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]) != cudaSuccess) { cudaGetLastError(); continue; }
        if (out) {
            snprintf(out[n].name, sizeof(out[n].name), "%s", ctx->mark_name[i]);
            out[n].round = ctx->mark_round[i];
            out[n].ms = ms;
            algo_bytes(ctx, ctx->mark_name[i], ctx->mark_round[i], &out[n].algo_bytes, &out[n].strict_bytes);
        }
        ++n;
    }
    return n;
}
