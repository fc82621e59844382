/*
 * gseg.h -- C-ABI of the B200-native graph-segmentation engine (libgseg.so).
 *
 * Drop-in boundary for the segmentation hot path of
 * akankshabaranwal/graph-algorithm-image-segmentation-GPGPU.  The mounted reference holds no source
 * (SURVEY.md section 0), so no reference header can be cited line by line; each entry point cites the
 * reference *stage* it replaces (Report.pdf page / section) and the parameter list BASELINE.json's
 * north_star fixes: input image, sigma, k, min_size, hierarchy level -> label image + hierarchy.
 * The closest published signature is F&H `segment`'s
 *     image<rgb>* segment_image(image<rgb>* im, float sigma, float c, int min_size, int* num_ccs)
 * (Report.pdf ref [23], the report's CPU baseline, p4 "Baseline"), which gseg_segment + gseg_labels
 * replace.
 *
 * Conventions: plain pointers and sizes only; 0 = success, negative = gseg_status; nothing throws
 * across the boundary; the caller owns every input/output buffer, the context owns all device
 * scratch.  gseg_create allocates everything the FELZ / HIER paths with sigma <= 2 need; the buffers
 * only some paths use (superpixel colour sums, the wide-sigma blur plane, the second label staging
 * buffer) are allocated by gseg_reserve, or on the first call that needs them when gseg_reserve was
 * not called -- after that nothing allocates inside gseg_segment.  One context per GPU per host
 * thread, contexts are independent and not thread-safe.  There is no CPU fallback: every entry
 * point that computes requires a CUDA device and fails with GSEG_E_CUDA otherwise.
 */
#ifndef GSEG_H
#define GSEG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSEG_VERSION 200

/* variant -- which reference branch's semantics to run (SURVEY.md section 2 rows 3-5) */
#define GSEG_FELZ 0     /* cuda-mst-naive: Boruvka + Felzenszwalb predicate + min-size (Report p2-3 s3.1) */
#define GSEG_HIER 1     /* fastmst_segment: one hierarchy level per Boruvka round, no predicate (p3-4 s3.2.2-3) */
#define GSEG_SUPERPIX 2 /* superpixel_gpu: per-round re-weighting by Sobel strength x mean colour (p4 s3.2.4) */

#define GSEG_MEM_HOST 0
#define GSEG_MEM_DEVICE 1

/* flags */
#define GSEG_FLAG_HOST_LOOP 1u /* host-driven schedule: one kernel per phase and a read-back per round (the
                                  reference's "ab conventional" driver, Report p3); used for per-kernel timing.
                                  Default (0): the device-resident round state drives every kernel, the host
                                  enqueues the whole run without reading anything back, and all small rounds
                                  run inside one persistent thread-block-cluster kernel. */

#define GSEG_FLAG_NO_DEDUP 2u  /* do not eliminate duplicate edges between rounds (measurement / A-B only: results are
                                  identical either way, see csrc/gseg_dedup.cuh) */

typedef enum gseg_status {
    GSEG_OK = 0,
    GSEG_E_ARG = -1,     /* bad argument (null pointer, size, connectivity, variant, sigma range) */
    GSEG_E_CUDA = -2,    /* CUDA runtime error or no device; gseg_last_error() has the text */
    GSEG_E_SIZE = -3,    /* image larger than the context was created for */
    GSEG_E_ARENA = -4,   /* supervertex-map arena exhausted (pathological round count) */
    GSEG_E_INTERNAL = -5, /* device-side watchdog tripped */
    GSEG_E_STATE = -6,   /* result requested before a successful gseg_segment */
    GSEG_E_LEVEL = -7,   /* hierarchy level out of range */
    GSEG_E_UNSUPPORTED = -8, /* optional dependency missing at run time (nvJPEG for gseg_segment_jpeg) */
    GSEG_E_RANGE = -9    /* label element type too narrow for the number of components / output buffer too small */
} gseg_status;

/* Parameters of one segmentation (BASELINE.json north_star: sigma, k, min_size, hierarchy level). */
typedef struct gseg_params {
    float sigma;          /* Gaussian pre-filter (Report p2 s2.1; p3 s3.2 par.2); 0 < 4*sigma+1 <= 64 taps */
    float k;              /* Felzenszwalb scale parameter (Report p2 par.1); FELZ only */
    int32_t min_size;     /* min-size post-merge (Report p3 step 6 "post-processing"); FELZ only */
    int32_t connectivity; /* 4 or 8 (BASELINE.json configs[1], configs[2]) */
    int32_t variant;      /* GSEG_FELZ | GSEG_HIER | GSEG_SUPERPIX */
    int32_t max_levels;   /* HIER/SUPERPIX: stop after this many levels; 0 = until one component */
    int32_t max_rounds;   /* cap on Boruvka rounds (Report p5: 10-20 in practice); 0 = 48 */
    uint32_t flags;
} gseg_params;

/* One row per executed Boruvka round (SURVEY.md section 5 "metrics": V_r, E_r per round). */
typedef struct gseg_round_stat {
    int64_t n_components; /* components entering the round */
    int64_t n_edges;      /* live (inter-component) edges of the list entering the round.  Until duplicates have been
                             dropped (n_edges_dedup == 0) this is every parallel edge, i.e. the count a plain
                             Boruvka contraction carries */
    int64_t n_merged;     /* components merged away by the round */
    int32_t phase;        /* 0 = predicate / hierarchy round, 1 = min-size round */
    int32_t in_tail;      /* 1 when the round ran inside the single-cluster tail kernel */
    float us_end;         /* device clock at the end of the round, microseconds since round 0's graph kernel started */
    float us_S, us_R, us_E; /* tail rounds: duration of the choose/scan, flatten and edge phases (else 0) */
    int32_t n_pages;      /* pages of the edge list entering the round */
    int32_t n_edges_dedup; /* != 0: duplicates have been dropped from the list this round ran on (by the sort step in front of
                              this round or of an earlier one); the edges it ran on */
} gseg_round_stat;

typedef struct gseg_ctx gseg_ctx;

int gseg_version(void);
/* sizeof of gseg_params, gseg_round_stat, gseg_kernel_time, gseg_pool_job, gseg_pool_result (in this order), so that a
 * binding (ctypes, cgo, JNI ...) can check its mirrors of the structs; returns how many there are. */
int gseg_abi_sizes(int32_t *out, int cap);
const char *gseg_strerror(int status);
const char *gseg_last_error(const gseg_ctx *ctx);

/* Replaces: per-branch main() device/scratch set-up (SURVEY.md section 1 L5/L4).  Allocates every
 * device buffer for images up to max_w x max_h on CUDA device `device`. */
int gseg_create(gseg_ctx **out, int device, int max_w, int max_h);
/* Same with the largest connectivity (4 or 8) the context will be used with: a 4-connected-only context
 * needs half the edge-list memory (a 32768 x 32768 image fits one B200 that way).  gseg_create = 8. */
int gseg_create_ex(gseg_ctx **out, int device, int max_w, int max_h, int max_connectivity);
void gseg_destroy(gseg_ctx *ctx);

/* Optional buffers, allocated up front instead of on first use (an allocation synchronises the whole
 * device and stalls the other contexts of a pool): caps = OR of GSEG_CAP_*. */
#define GSEG_CAP_SUPERPIX 1u   /* colour sums + means + Sobel plane of the superpixel variant */
#define GSEG_CAP_WIDE_SIGMA 2u /* intermediate plane of the general blur (more than 8 one-sided taps) */
#define GSEG_CAP_LEVELS 4u     /* second staging buffer of gseg_labels_all / gseg_colorize to host memory */
#define GSEG_CAP_JPEG 8u       /* buffers of the in-house JPEG decoder (staged file, coefficients, sample planes) */
#define GSEG_CAP_REGIONS 16u   /* gseg_regions / gseg_render scratch: a table of 64 bytes per pixel (host output of tables
                                  with more than (max_w*max_h + 64)/8 records) and the staging of host-memory input */
int gseg_reserve(gseg_ctx *ctx, uint32_t caps);

/* Pinned host memory for inputs/outputs of the asynchronous calls (cudaHostAlloc behind a plain pointer, so a
 * C/C++ caller needs no CUDA headers). */
void *gseg_host_alloc(size_t bytes);
/* Write-combined pinned memory: for INPUT buffers the CPU only writes (reading it from the CPU is very slow); the
 * device's reads do not snoop the CPU caches. */
void *gseg_host_alloc_wc(size_t bytes);
void gseg_host_free(void *p);

/* Run the context's work on a caller-owned CUDA stream (cudaStream_t as void*); NULL = own stream. */
int gseg_set_stream(gseg_ctx *ctx, void *cuda_stream);
void *gseg_get_stream(const gseg_ctx *ctx); /* the cudaStream_t the context's work is enqueued on */

/* Scheduling knob (no effect on results): a Boruvka round whose graph has at most max_edges live edges
 * and max_components components runs inside the single-cluster tail kernel instead of grid-wide
 * kernels.  (0, 0) disables the tail.  Defaults: 262144 edges, 65536 components. */
int gseg_set_tail(gseg_ctx *ctx, uint32_t max_edges, uint32_t max_components);

/* Scheduling knob (no effect on results): CTAs of the tail kernel's thread-block cluster (1..16, default 16 = lowest latency of
 * one image alone; a pool of >= 4 contexts uses 8, which leaves more SMs to the other images' grid-wide kernels).
 * gseg_tail_cluster returns the size in use; gseg_tail_cluster_from_env is 1 when GSEG_TAIL_CLUSTER set it. */
int gseg_set_tail_cluster(gseg_ctx *ctx, int ctas);
int gseg_tail_cluster(const gseg_ctx *ctx);
int gseg_tail_cluster_from_env(const gseg_ctx *ctx);

/* Scheduling knob (no effect on results): resident blocks per SM the grid-wide kernels are sized for
 * (1..8, default 4).  With several contexts in flight per GPU, 2 leaves room for their kernels to overlap. */
int gseg_set_blocks_per_sm(gseg_ctx *ctx, int blocks);

/* Duplicate-edge elimination between rounds (SURVEY.md section 8a row a10; the reference's DPP branches sort the packed
 * edge keys every round and keep the lightest of every run of duplicates, Report.pdf p3 s3.2.2).  FELZ / HIER runs sort
 * the list by component pair with the in-house onesweep radix sort once the graph has at most max_components components
 * (default 4096, at most 65536) while the list still holds >= min_edges edges (default 2^19) and >= min_ratio edges per
 * component (default 8); they keep the minimum (weight, list position) of every run and re-compact the list in order
 * (0 = keep the current value of a threshold).  The result is identical either way; the thresholds are where the sort
 * costs less than the rounds it shortens on B200 (DESIGN.md has the A/B).  GSEG_DEDUP=0 in the environment switches it
 * off for every context of the process, GSEG_DEDUP_V / GSEG_DEDUP_MIN / GSEG_DEDUP_RATIO set the thresholds. */
int gseg_set_dedup(gseg_ctx *ctx, int on, uint32_t min_edges, uint32_t min_ratio, uint32_t max_components);

/* Replaces: L3 pre-filter + L2 graph creation + L1 segmentation core of one reference executable
 * (Report p2 Fig.1; p3 s3.2.1; p2-3 s3.1 steps 1-9; p3-4 s3.2.2; p4 s3.2.4).
 * rgb: interleaved 8-bit RGB, `stride_bytes` per row (>= 3*w), in host or device memory (mem_kind).
 * Returns when the partition is complete on the device. */
int gseg_segment(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride_bytes, int mem_kind,
                 const gseg_params *params);

/* Asynchronous form: enqueue only (host input must be pinned and stay valid); gseg_wait completes it. */
int gseg_segment_async(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride_bytes, int mem_kind,
                       const gseg_params *params);
int gseg_wait(gseg_ctx *ctx);

/* Number of hierarchy levels produced (FELZ: 1).  Replaces: the stored per-round supervertex ids
 * (Report p4 s3.2.3 par.1). */
int gseg_num_levels(const gseg_ctx *ctx);
/* Components at `level` (0-based; -1 = last). */
int gseg_num_components(const gseg_ctx *ctx, int level);

/* Replaces: L0 hierarchy materialisation, one thread per pixel mapping the previous level's ids
 * through the stored supervertex ids (Report p4 s3.2.3).  out: w*h int32, row-major, dense ids in
 * [0, gseg_num_components(level)).  level -1 = last level / the FELZ partition. */
int gseg_labels(gseg_ctx *ctx, int level, int32_t *out, int mem_kind);
/* Asynchronous form of gseg_labels: enqueues the materialisation (and the copy to pinned host memory) on
 * the context's stream and returns; gseg_sync (or any later synchronous call) completes it. */
int gseg_labels_async(gseg_ctx *ctx, int level, int32_t *out, int mem_kind);
int gseg_sync(gseg_ctx *ctx);

/* The same label image in a narrower element type: elem_bytes = 4 (int32), 2 (uint16) or 1 (uint8).  Lossless:
 * GSEG_E_RANGE when gseg_num_components(level) does not fit the type.  gseg_label_bytes returns the narrowest
 * of 1, 2, 4 that holds `level`.  A 1080p FELZ partition has ~10^2 components: its label image leaves the GPU
 * in 2 MB instead of 8 (the device->host copy is the larger half of an end-to-end run's PCIe bytes). */
int gseg_label_bytes(const gseg_ctx *ctx, int level);
int gseg_labels_ex(gseg_ctx *ctx, int level, void *out, int elem_bytes, int mem_kind);
int gseg_labels_ex_async(gseg_ctx *ctx, int level, void *out, int elem_bytes, int mem_kind);

/* The hierarchy in its stored form -- the per-round supervertex ids the reference keeps and materialises on
 * demand (Report p4 s3.2.3 par.1): out[offsets[l] + i] = id at level l of component i of level l-1 (level -1 =
 * pixels, so the first w*h entries are the level-0 label image); offsets[n_levels] = entries written.  Returns
 * n_levels (HIER / SUPERPIX; FELZ: 1 level = the final label image).  GSEG_E_RANGE when cap_entries or
 * cap_offsets (needs n_levels + 1) is too small; call with out = NULL to get the sizes. */
int gseg_hierarchy(gseg_ctx *ctx, uint32_t *out, int64_t cap_entries, int64_t *offsets, int cap_offsets, int mem_kind);
int gseg_hierarchy_async(gseg_ctx *ctx, uint32_t *out, int64_t cap_entries, int64_t *offsets, int cap_offsets, int mem_kind);

/* All levels 0..n-1 in one pass (level l at out + l*w*h); n = min(max_levels, gseg_num_levels). */
int gseg_labels_all(gseg_ctx *ctx, int32_t *out, int max_levels, int mem_kind);

/* Replaces: random colour table + colour image (cuRAND, Report p4 s3.2.3).  out: w*h*3 bytes. */
int gseg_colorize(gseg_ctx *ctx, int level, uint64_t seed, uint8_t *out_rgb, int mem_kind);

/* Per-component statistics of `level` (same level rules as gseg_labels_ex; component c = dense label c):
 * out[8*c + 0..7] = count, sum r, sum g, sum b (the INPUT image's 8-bit channels), sum x, sum y,
 * x0 | y0 << 32 (bounding-box minimum, inclusive), x1 | y1 << 32 (maximum, inclusive) -- n = gseg_num_components(level)
 * records of 64 bytes, all integers (DESIGN.md section 2 item 10).  The input is `rgb` (stride_bytes per row, host or
 * device memory as rgb_mem_kind says), or with rgb == NULL the image the context staged (host input or JPEG;
 * GSEG_E_STATE when the run read caller-owned device memory).  GSEG_E_STATE after an explicit-graph run or a joined
 * strip, GSEG_E_RANGE when cap_records < n, GSEG_E_ARG for device output that is not 8-byte aligned.  Returns n. */
int gseg_regions_async(gseg_ctx *ctx, int level, const uint8_t *rgb, int stride_bytes, int rgb_mem_kind, uint64_t *out,
                       int64_t cap_records, int mem_kind);
int gseg_regions(gseg_ctx *ctx, int level, const uint8_t *rgb, int stride_bytes, int rgb_mem_kind, uint64_t *out,
                 int64_t cap_records, int mem_kind); /* blocking form */

/* Pictures of `level` (blocking).  A boundary pixel has at least one 4-neighbour inside the image with another label.
 * MEAN and OVERLAY read the input like gseg_regions (rgb == NULL: the staged image); BOUNDARY ignores rgb. */
#define GSEG_RENDER_MEAN 0     /* every pixel = its region's rounded mean colour (sum + count/2) / count; out: w*h*3 bytes */
#define GSEG_RENDER_OVERLAY 1  /* input pixels, boundary pixels set to `colour` (0xRRGGBB); out: w*h*3 bytes             */
#define GSEG_RENDER_BOUNDARY 2 /* 1 byte per pixel: 1 = boundary pixel, 0 = not; out: w*h bytes                           */
int gseg_render(gseg_ctx *ctx, int level, int mode, uint32_t colour, const uint8_t *rgb, int stride_bytes, int rgb_mem_kind,
                uint8_t *out, int mem_kind);

/* Round-0 edge weights in edge-index order idx = d*w*h + (y*w+x), d in 0..D-1, D = 2 (E,S) or 4 (E,S,SE,NE);
 * +inf where the edge does not exist (SUPERPIX: the static edge strength).  For the 1e-6 check. */
int gseg_weights(gseg_ctx *ctx, float *out, int mem_kind);
/* Blurred image, 3 planes of w*h floats (R,G,B). */
int gseg_blurred(gseg_ctx *ctx, float *out, int mem_kind);

/* ---- tiled schedule (BASELINE.json configs[4], north_star: "cross-tile boundary edges exchanged over
 * NVLink via NCCL before the final Boruvka rounds"; DESIGN.md "Tiled schedule") ------------------------
 * A strip is segmented like any image; its final component graph is exported, the strips' graphs are
 * joined by the cut edges on the host side of the exchange, and the joined graph runs the same rounds.
 *
 * gseg_export_graph: components (size, Int(C)) and live inter-component edges (a, b, weight; ids = the
 * dense labels of gseg_labels(-1); list order = edge-index order) of the last FELZ/HIER run.  Call with
 * NULL arrays to get the counts, then with host arrays of at least that capacity.
 * dedup != 0: parallel edges between the same two components are reduced to their minimum (weight, list
 * position) -- the reference's sort-based duplicate elimination (Report p3 s3.2.2), on the in-house
 * onesweep radix sort; the partition the joined rounds produce is unchanged, the list is ~100x shorter. */
int gseg_export_graph(gseg_ctx *ctx, int dedup, int64_t *n_components, int64_t *n_edges, uint32_t *size, float *Int,
                      uint32_t *ea, uint32_t *eb, float *w, int64_t cap_components, int64_t cap_edges);
/* Rows y0 .. y0+nrows-1 of the blurred planes: out[3][nrows][w] (the cut-edge weights need the boundary rows). */
int gseg_blurred_rows(gseg_ctx *ctx, int y0, int nrows, float *out, int mem_kind);
/* The Boruvka rounds of `params->variant` (FELZ or HIER) on an explicit graph in host memory: components
 * with (size, Int), edges (ea, eb, w) whose list position is the tie-break.  labels_out[c] = dense final
 * component of input component c; returns the number of final components (or a negative status). */
int gseg_segment_graph(gseg_ctx *ctx, int64_t n_components, const uint32_t *size, const float *Int, int64_t n_edges,
                       const uint32_t *ea, const uint32_t *eb, const float *w, const gseg_params *params,
                       int32_t *labels_out);

/* ---- tiled schedule, device side (no host bounce: the exchange is an all-gather of device buffers) ----------
 * gseg_segment_strip_async: one horizontal strip of a larger image.  `rgb` points at the first row of a buffer
 *   holding halo_top rows above the strip, the strip's h rows, and halo_bottom rows below it; with halo >=
 *   ceil(4 sigma) rows on every side that has a neighbour strip, the strip's blurred pixels and hence all of
 *   its edge weights (and the cut edges') are bit-identical to the untiled image's (SURVEY.md section 8e
 *   "4-row input halo").  The graph covers the strip's h rows only.  FELZ / HIER.
 * gseg_strip_record: what a strip contributes to the exchange, written to DEVICE memory as 32-bit words:
 *   header[8] = {magic, nV, nE, w, 0, 0, 0, 0} | (size, Int bits)[nV] | (a, b)[nE] | weight bits[nE] |
 *   labels of the first row [w] | of the last row [w] | blurred colours of the first row [3][w] | last row [3][w].
 *   dev_out = NULL: only *bytes is set.  Keeps the strip's dense label image in the context.
 * gseg_join_segment: `dev_records` = n_strips records (strip order = top to bottom) at a distance of
 *   record_stride_bytes (the output of an all-gather of equal-size buffers).  Joins them on the device --
 *   components renumbered strip by strip; list = strip 0's edges, cut edges 0|1 (S, then SE, NE; weights from the
 *   two blurred boundary rows), strip 1's edges, ... -- runs the rounds of params->variant on the joined graph and
 *   writes the final label image of strip `my_strip` (image-global dense ids; elem_bytes 1/2/4 as in
 *   gseg_labels_ex; labels_out may be NULL).  Returns the number of final components. */
int gseg_segment_strip_async(gseg_ctx *ctx, const uint8_t *rgb, int w, int h, int stride_bytes, int mem_kind, int halo_top,
                             int halo_bottom, const gseg_params *params);
int gseg_strip_record(gseg_ctx *ctx, int dedup, void *dev_out, int64_t cap_bytes, int64_t *bytes);
int gseg_join_segment(gseg_ctx *ctx, const void *dev_records, int n_strips, int64_t record_stride_bytes, int my_strip,
                      const gseg_params *params, void *labels_out, int elem_bytes, int mem_kind, int64_t *n_joined_components,
                      int64_t *n_joined_edges);

/* ---- JPEG input decoded on the GPU (SURVEY.md section 8f N2) --------------------------------------
 * The reference's batch benchmark reads a JPEG data set through cv::imread on the host (README.md:26).
 * Here the compressed bytes go to the GPU (7-10x fewer bytes over PCIe than the RGB image) and are decoded
 * there into the context's staged RGB buffer, on the context's stream, in front of the blur; the decoded
 * image never visits the host.  Two decoders:
 *   GSEG_JPEG_OWN     hand-written kernels (csrc/gseg_jpeg.cuh): baseline / extended-sequential Huffman,
 *                     8-bit, grey or YCbCr, luma 1x1 / 2x1 / 1x2 / 2x2 / 4x1, one interleaved scan.  The
 *                     pixels are bit-identical to libjpeg's default decoder (islow IDCT, fancy upsampling),
 *                     i.e. to what cv::imread gives the reference.  Files with short restart intervals
 *                     (<= 8 MCUs; cv::IMWRITE_JPEG_RST_INTERVAL, jpegtran -restart): one thread per
 *                     interval, the lowest latency (1080p: 0.15-0.8 ms).  Files without restart markers or
 *                     with longer intervals: self-synchronising sub-sequences in one thread-block cluster
 *                     (1080p: ~1.2 ms).
 *   GSEG_JPEG_NVJPEG  nvJPEG (CUDA toolkit library, loaded with dlopen on first use -- libgseg.so does not
 *                     link it): everything else it can decode (progressive ...); Huffman stage on the host.
 *   GSEG_JPEG_AUTO    (default) OWN for every file it supports, NVJPEG otherwise.
 *   gseg_jpeg_info          width / height of a JPEG (host only: parses the header, needs no device).
 *   gseg_segment_jpeg_async decode + enqueue the segmentation (complete it with gseg_wait, or use
 *   gseg_segment_jpeg       the blocking form); *w, *h receive the image size.
 *   gseg_set_jpeg_backend / gseg_jpeg_backend_used   choose the decoder / which one the last JPEG run used.
 *   gseg_input_rgb          the interleaved RGB image the last run read, when it was staged by the
 *                           context (host input or JPEG); GSEG_E_STATE for caller-owned device input.
 * GSEG_E_ARG for data that is no JPEG or does not decode (corrupt entropy-coded data is reported by
 * gseg_wait), GSEG_E_UNSUPPORTED when the file needs nvJPEG and libnvjpeg cannot be loaded, or when
 * GSEG_JPEG_OWN was forced for a file the in-house decoder does not take. */
#define GSEG_JPEG_AUTO 0
#define GSEG_JPEG_OWN 1
#define GSEG_JPEG_NVJPEG 2
int gseg_jpeg_info(const void *jpeg, size_t nbytes, int *w, int *h);
int gseg_segment_jpeg_async(gseg_ctx *ctx, const void *jpeg, size_t nbytes, const gseg_params *params, int *w, int *h);
int gseg_segment_jpeg(gseg_ctx *ctx, const void *jpeg, size_t nbytes, const gseg_params *params, int *w, int *h);
int gseg_input_rgb(gseg_ctx *ctx, uint8_t *out_rgb, int mem_kind);
/* The decode alone (in-house decoder only): interleaved RGB, tightly packed, into caller-owned DEVICE memory on a
 * caller-chosen stream (NULL = the context's).  The batch pipeline uses it to decode a context's next image on its copy
 * stream while the current one is still being segmented.  The context's next gseg_segment_async (give it rgb_out_device
 * as GSEG_MEM_DEVICE input, ordered behind the decode) reports corrupt entropy-coded data through gseg_wait.
 * GSEG_E_UNSUPPORTED when the file needs nvJPEG under the context's backend setting, GSEG_E_RANGE when it does not fit. */
int gseg_jpeg_decode_async(gseg_ctx *ctx, const void *jpeg, size_t nbytes, uint8_t *rgb_out_device, size_t out_capacity,
                           void *cuda_stream, int *w, int *h);
int gseg_set_jpeg_backend(gseg_ctx *ctx, int backend);
int gseg_jpeg_backend_used(const gseg_ctx *ctx);

/* Per-round statistics of the last run; returns number of rounds (<= cap written). */
int gseg_stats(const gseg_ctx *ctx, gseg_round_stat *out, int cap);

/* Deterministic synthetic input (SURVEY.md section 8d): w*h*3 bytes into host or device memory. */
int gseg_synth(gseg_ctx *ctx, uint8_t *out_rgb, int w, int h, uint64_t seed, int mem_kind);
/* Rows [y_first, y_first + nrows) of the synthetic image of width w and the same seed (a pixel depends on its
 * coordinates and the seed only): strips of the gigapixel image are generated where they are segmented. */
int gseg_synth_rows(gseg_ctx *ctx, uint8_t *out_rgb, int w, int y_first, int nrows, uint64_t seed, int mem_kind);

/* Measurement support (SURVEY.md section 5 "tracing"; section 8d): with profiling on, the host-driven
 * schedule brackets every kernel with CUDA events on the context's stream. */
typedef struct gseg_kernel_time {
    char name[24];
    int32_t round;
    float ms;
    double algo_bytes;   /* algorithmic bytes of this launch: SURVEY.md section 8(d) accounting -- every input array read
                            once, every output written once, gathers at element size, one 8-byte minimum per component
                            (not per atomic) -- see DESIGN.md "Kernels" */
    double strict_bytes; /* the same with every gathered array counted once however often it is gathered */
} gseg_kernel_time;
int gseg_set_profiling(gseg_ctx *ctx, int on);
int gseg_profile_read(gseg_ctx *ctx, gseg_kernel_time *out, int cap);
/* Kernels launched by this context since creation (graph replays count their kernel nodes). */
long long gseg_launch_count(const gseg_ctx *ctx);
/* Arena compactions since creation (FELZ runs whose per-round maps outgrew the arena were folded and resumed). */
long long gseg_compaction_count(const gseg_ctx *ctx);

/* ---- batch pipeline (the reference's loop over the images of its performance data set, Report.pdf p4 s4.1;
 * README.md:26-28) ---------------------------------------------------------------------------------------
 * A pool owns n_contexts contexts (one CUDA stream each) on one GPU and keeps them in flight: job t runs on
 * context t mod n_contexts, a context gets its next job as soon as its previous one is complete, the output
 * copy of a job is ordered before the next job of its context, and results come back in submission order.
 * Inputs and outputs of asynchronous copies should be pinned (gseg_host_alloc); an input must stay valid until
 * the job's result has been returned.  Not thread-safe: call a pool from one host thread.
 *   gseg_pool_submit  enqueue one job (may first wait for the previous job of the same context)
 *   gseg_pool_next    the oldest job's result, its output complete in job.out (GSEG_E_STATE: nothing in flight)
 *   gseg_pool_run     a whole batch: n submits, n results (results[i] belongs to jobs[i])
 *   gseg_pool_copy_ceiling  the batch's host<->device copies alone (same buffers, bytes and streams, no
 *                     kernels), ms per batch: what the box's PCIe / host memory allows for this batch */
#define GSEG_OUT_NONE 0      /* nothing leaves the context (results stay there until its next job) */
#define GSEG_OUT_LABELS 1    /* label image of `level`; elem_bytes 0 = the narrowest lossless type, else 1 / 2 / 4 */
#define GSEG_OUT_HIERARCHY 2 /* the stored hierarchy (gseg_hierarchy): level-0 labels + one map per further level */
#define GSEG_OUT_REGIONS 3   /* label image of `level` as GSEG_OUT_LABELS, then at the next 64-byte-aligned offset the region
                                table (gseg_regions) of the job's input: offsets[0] = 0, offsets[1] = the table's byte offset,
                                offsets[2] = out_bytes = the end */
#define GSEG_POOL_MAXLEVELS 64
typedef struct gseg_pool gseg_pool;
typedef struct gseg_pool_job {
    const void *input;    /* interleaved 8-bit RGB, or a JPEG file's bytes when jpeg_bytes != 0 */
    size_t jpeg_bytes;
    int32_t w, h, stride_bytes /* 0 = 3*w */, mem_kind;
    gseg_params params;
    int32_t out_mode, level, elem_bytes, out_mem_kind;
    void *out;
    size_t out_capacity;  /* bytes */
    void *user;           /* returned with the result */
} gseg_pool_job;
typedef struct gseg_pool_result {
    int64_t ticket;       /* submission index */
    int32_t status;       /* gseg_status of the job */
    int32_t w, h, n_levels, n_components /* at job.level */, elem_bytes;
    int64_t out_bytes;    /* bytes written to job.out */
    int64_t offsets[GSEG_POOL_MAXLEVELS + 1]; /* GSEG_OUT_HIERARCHY: gseg_hierarchy's offsets */
    void *out, *user;
} gseg_pool_result;
int gseg_pool_create(gseg_pool **out, int device, int max_w, int max_h, int max_connectivity, int n_contexts, uint32_t caps);
void gseg_pool_destroy(gseg_pool *pool);
int gseg_pool_contexts(const gseg_pool *pool);
gseg_ctx *gseg_pool_context(gseg_pool *pool, int i);
int gseg_pool_pending(const gseg_pool *pool);
const char *gseg_pool_last_error(const gseg_pool *pool);
int gseg_pool_submit(gseg_pool *pool, const gseg_pool_job *job, int64_t *ticket);
int gseg_pool_next(gseg_pool *pool, gseg_pool_result *out);
int gseg_pool_run(gseg_pool *pool, const gseg_pool_job *jobs, int n, gseg_pool_result *results);
int gseg_pool_copy_ceiling(gseg_pool *pool, const gseg_pool_job *jobs, const gseg_pool_result *results, int n, int reps,
                           double *ms_per_batch);

/* Stand-alone primitives of the edge-dedup path (SURVEY.md section 8a row a10; Report p3 s3.2.2
 * "sort"): in-house onesweep radix sort of 64-bit keys with 32-bit payload, on device memory. */
/* Runs on the context's stream and returns when the arrays are sorted; keys / vals must be complete when it is
 * called (work enqueued on other streams is not waited for). */
int gseg_sort_pairs_u64(gseg_ctx *ctx, uint64_t *keys, uint32_t *vals, int64_t n, int begin_bit, int end_bit);

#ifdef __cplusplus
}
#endif
#endif /* GSEG_H */
