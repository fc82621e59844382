// gseg_pool.cu -- batch pipeline over the C-ABI of include/gseg.h (gseg_pool_*).
//
// The reference times a loop over the images of its performance data set, one image at a time on one
// stream (Report.pdf p4 s4.1; README.md:26-28).  Here S contexts (one CUDA stream each) stay in flight on one
// GPU: the latency-bound late Boruvka rounds of one image (a single thread-block cluster) overlap the
// bandwidth-bound early rounds of the next ones, and the host->device copy of an image and the device->host
// copy of a label image overlap the kernels of the other contexts.  Rolling schedule: job t runs on context
// t mod S; a context gets its next job as soon as its previous one is complete, its output copy is ordered on
// the context's stream before the next job's kernels, and results are handed out in submission order.
//
// Host code only: everything that computes is a gseg_* call on a context.  No thread is created: the pool
// advances inside gseg_pool_submit / gseg_pool_next on the caller's thread (contexts are not thread-safe).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <deque>
#include <new>
#include <vector>

#include "../../include/gseg.h"

namespace {

struct Rec {
    gseg_pool_job job;
    gseg_pool_result res;
    int slot;
    bool running;       // the segmentation has been enqueued but not waited for
    const uint8_t *rgb; // GSEG_OUT_REGIONS: the device image the job read (nullptr: the context staged it itself)
    int rgb_stride;
    int stage_b;        // ... which is pool staging buffer stage[stage_b] (-1: it is not)
    cudaEvent_t ev;     // completion of the output copy (nullptr: nothing was enqueued)
};

} // namespace

struct gseg_pool {
    int device, S;
    size_t stage_bytes;    // capacity of one input staging buffer (max_w * max_h * 3)
    std::vector<gseg_ctx *> ctx;
    // Input prefetch: every context has two device staging buffers and a copy stream.  The host->device copy of a job is
    // issued BEFORE the pool waits for the context's previous job, into the buffer that job is not reading, so it runs
    // under that job's kernels instead of in front of its own (SURVEY.md section 8e "pinned double-buffered H2D").
    std::vector<cudaStream_t> copy_stream;
    std::vector<uint8_t *> stage;      // [2 * S]
    std::vector<cudaEvent_t> stage_ev; // [2 * S]
    std::vector<int> stage_next;       // per context: which of its two buffers the next job takes
    // 1: a GSEG_OUT_REGIONS job's statistics kernel reads stage[b] on the context's stream after its segmentation was
    // waited for, and stage_ev[b] was re-recorded behind it there: the next write into stage[b] (host copy or JPEG decode,
    // on the copy stream) waits for that event first.  Without it, jpeg_prefetch would decode job t + 2S into the buffer
    // while job t's k_regions (enqueued by retire in the submit of job t + S) may still be reading it.
    std::vector<int> stage_read;       // [2 * S]
    // JPEG jobs: the decode of a context's NEXT job (in-house kernels, on the copy stream, into the free staging buffer) is
    // enqueued as soon as the current one has been submitted -- a whole pipeline turn ahead (gseg_pool_run knows the job)
    struct Pref { const void *input; size_t bytes; int w, h, b; bool valid; };
    std::vector<Pref> pref; // per context
    std::vector<int> busy; // per context: 1 while its last job has not been retired
    std::deque<Rec> q;     // submission order
    std::vector<cudaEvent_t> free_ev;
    int64_t next_ticket;
    char err[256];
};

static cudaEvent_t take_event(gseg_pool *p) {
    if (!p->free_ev.empty()) { cudaEvent_t e = p->free_ev.back(); p->free_ev.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return e;
}

extern "C" int gseg_pool_create(gseg_pool **out, int device, int max_w, int max_h, int max_connectivity, int n_contexts,
                                uint32_t caps) {
    if (!out || n_contexts < 1 || n_contexts > 64) return GSEG_E_ARG;
    *out = nullptr;
    gseg_pool *p = new (std::nothrow) gseg_pool();
    if (!p) return GSEG_E_ARG;
    p->device = device; p->S = n_contexts; p->next_ticket = 0; p->err[0] = 0;
    p->stage_bytes = (size_t)max_w * (size_t)max_h * 3;
    int rc = GSEG_OK;
    for (int i = 0; i < n_contexts && !rc; ++i) {
        gseg_ctx *c = nullptr;
        rc = gseg_create_ex(&c, device, max_w, max_h, max_connectivity);
        if (!rc) {
            p->ctx.push_back(c);
            p->busy.push_back(0);
            p->stage_next.push_back(0);
            p->pref.push_back(gseg_pool::Pref{nullptr, 0, 0, 0, 0, false});
            cudaStream_t cs = nullptr;
            if (cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking) != cudaSuccess) rc = GSEG_E_CUDA;
            p->copy_stream.push_back(cs);
            for (int b = 0; b < 2 && !rc; ++b) {
                uint8_t *d = nullptr;
                cudaEvent_t e = nullptr;
                if (cudaMalloc((void **)&d, p->stage_bytes + 64) != cudaSuccess || cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) rc = GSEG_E_CUDA;
                p->stage.push_back(d);
                p->stage_ev.push_back(e);
                p->stage_read.push_back(0);
            }
            if (caps) rc = gseg_reserve(c, caps);
            // several contexts share the SMs: size every grid for 2 resident blocks per SM so that kernels of
            // different images run side by side (measured in round 1: +12 % over 4 with 8 contexts)
            int bps = 2;
            if (const char *ev = getenv("GSEG_POOL_BLOCKS_PER_SM")) bps = atoi(ev) >= 1 && atoi(ev) <= 8 ? atoi(ev) : 2;
            if (!rc && n_contexts >= 4) rc = gseg_set_blocks_per_sm(c, bps);
            // ... and the tail cluster takes 8 SMs instead of 16: a tail CTA (1024 threads x 64 registers) owns its SM, and
            // with eight images in flight three to four tails are running at any time -- at 16 CTAs each they hold a third of
            // the GPU for latency-bound work (measured: 9 298 -> 9 686 Mpixel/s; 4 CTAs 9 619, 2 CTAs 8 881)
            if (!rc && n_contexts >= 4 && !gseg_tail_cluster_from_env(c)) rc = gseg_set_tail_cluster(c, 8);
        }
    }
    if (rc) { gseg_pool_destroy(p); return rc; }
    *out = p;
    return GSEG_OK;
}

extern "C" void gseg_pool_destroy(gseg_pool *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    for (gseg_ctx *c : p->ctx) { gseg_wait(c); gseg_sync(c); }
    for (Rec &r : p->q)
        if (r.ev) cudaEventDestroy(r.ev);
    for (cudaEvent_t e : p->free_ev) cudaEventDestroy(e);
    for (cudaStream_t cs : p->copy_stream) if (cs) { cudaStreamSynchronize(cs); cudaStreamDestroy(cs); }
    for (uint8_t *d : p->stage) cudaFree(d);
    for (cudaEvent_t e : p->stage_ev) if (e) cudaEventDestroy(e);
    for (gseg_ctx *c : p->ctx) gseg_destroy(c);
    delete p;
}

// sizeof of every struct that crosses the ABI, for bindings to check their mirrors against
extern "C" int gseg_abi_sizes(int32_t *out, int cap) {
    const int32_t v[5] = {(int32_t)sizeof(gseg_params), (int32_t)sizeof(gseg_round_stat), (int32_t)sizeof(gseg_kernel_time),
                          (int32_t)sizeof(gseg_pool_job), (int32_t)sizeof(gseg_pool_result)};
    for (int i = 0; i < 5 && i < cap && out; ++i) out[i] = v[i];
    return 5;
}

extern "C" int gseg_pool_contexts(const gseg_pool *p) { return p ? p->S : GSEG_E_ARG; }
extern "C" gseg_ctx *gseg_pool_context(gseg_pool *p, int i) { return p && i >= 0 && i < p->S ? p->ctx[(size_t)i] : nullptr; }
extern "C" int gseg_pool_pending(const gseg_pool *p) { return p ? (int)p->q.size() : GSEG_E_ARG; }
extern "C" const char *gseg_pool_last_error(const gseg_pool *p) { return p ? p->err : "null pool"; }

// The job's segmentation is complete on the device: read what the host needs to know, enqueue the output copy
// on the context's stream and mark its end with an event.  The context is free for its next job afterwards.
// A write into stage[b] on the copy stream of `slot` is about to be enqueued: order it behind a reader retire left.
static cudaError_t stage_claim(gseg_pool *p, int slot, int b) {
    if (!p->stage_read[(size_t)b]) return cudaSuccess;
    p->stage_read[(size_t)b] = 0;
    return cudaStreamWaitEvent(p->copy_stream[(size_t)slot], p->stage_ev[(size_t)b], 0);
}

static void retire(gseg_pool *p, Rec &r) {
    gseg_ctx *c = p->ctx[(size_t)r.slot];
    r.running = false;
    p->busy[(size_t)r.slot] = 0;
    gseg_pool_result &res = r.res;
    int rc = gseg_wait(c);
    if (rc) { res.status = rc; snprintf(p->err, sizeof(p->err), "job %lld: %s", (long long)res.ticket, gseg_last_error(c)); return; }
    res.n_levels = gseg_num_levels(c);
    res.n_components = gseg_num_components(c, r.job.level);
    if (res.n_components < 0) { res.status = res.n_components; return; }
    const size_t V = (size_t)res.w * res.h;
    if (r.job.out_mode == GSEG_OUT_LABELS) {
        const int need = gseg_label_bytes(c, r.job.level);
        const int eb = r.job.elem_bytes ? r.job.elem_bytes : need;
        if (!r.job.out || V * (size_t)eb > r.job.out_capacity) { res.status = GSEG_E_RANGE; return; }
        rc = gseg_labels_ex_async(c, r.job.level, r.job.out, eb, r.job.out_mem_kind);
        res.elem_bytes = eb; res.out_bytes = (int64_t)(V * (size_t)eb);
    } else if (r.job.out_mode == GSEG_OUT_REGIONS) {
        const int need = gseg_label_bytes(c, r.job.level);
        const int eb = r.job.elem_bytes ? r.job.elem_bytes : need;
        const size_t off = (V * (size_t)eb + 63) & ~(size_t)63, end = off + (size_t)res.n_components * 64;
        if (!r.job.out || end > r.job.out_capacity) { res.status = GSEG_E_RANGE; return; }
        rc = gseg_labels_ex_async(c, r.job.level, r.job.out, eb, r.job.out_mem_kind);
        if (!rc) {
            rc = gseg_regions_async(c, r.job.level, r.rgb, r.rgb_stride, GSEG_MEM_DEVICE, (uint64_t *)((uint8_t *)r.job.out + off),
                                    res.n_components, r.job.out_mem_kind);
            if (rc >= 0) rc = GSEG_OK;
        }
        if (!rc && r.stage_b >= 0) { // the staging buffer is read until here: see gseg_pool::stage_read
            cudaEventRecord(p->stage_ev[(size_t)r.stage_b], (cudaStream_t)gseg_get_stream(c));
            p->stage_read[(size_t)r.stage_b] = 1;
        }
        res.elem_bytes = eb; res.offsets[0] = 0; res.offsets[1] = (int64_t)off; res.offsets[2] = (int64_t)end;
        res.out_bytes = (int64_t)end;
    } else if (r.job.out_mode == GSEG_OUT_HIERARCHY) {
        rc = gseg_hierarchy_async(c, (uint32_t *)r.job.out, (int64_t)(r.job.out_capacity / 4), res.offsets, GSEG_POOL_MAXLEVELS + 1,
                                  r.job.out_mem_kind);
        if (rc > 0) { res.n_levels = rc; res.elem_bytes = 4; res.out_bytes = res.offsets[rc] * 4; rc = GSEG_OK; }
    }
    if (rc) { res.status = rc; snprintf(p->err, sizeof(p->err), "job %lld: %s", (long long)res.ticket, gseg_last_error(c)); return; }
    if (r.job.out_mode != GSEG_OUT_NONE) {
        r.ev = take_event(p);
        if (r.ev) cudaEventRecord(r.ev, (cudaStream_t)gseg_get_stream(c));
        else res.status = gseg_sync(c); // no event to be had: complete the copy now
    }
}

// Decode a JPEG job of context `slot` ahead of its submission: file bytes over PCIe + the in-house decoder's kernels on the
// context's copy stream, into the staging buffer the context's running job is not reading.  GSEG_E_UNSUPPORTED / GSEG_E_RANGE:
// the file goes the nvJPEG way at submission (nothing was enqueued).
static int jpeg_prefetch(gseg_pool *p, int slot, const gseg_pool_job *job) {
    gseg_pool::Pref &pf = p->pref[(size_t)slot];
    if (pf.valid) p->stage_next[(size_t)slot] = pf.b & 1; // a decode nobody came for: its buffer is free again
    pf.valid = false;
    gseg_ctx *c = p->ctx[(size_t)slot];
    const int b = 2 * slot + p->stage_next[(size_t)slot];
    int w = 0, h = 0;
    if (stage_claim(p, slot, b) != cudaSuccess) { cudaGetLastError(); return GSEG_E_CUDA; }
    const int rc = gseg_jpeg_decode_async(c, job->input, job->jpeg_bytes, p->stage[(size_t)b], p->stage_bytes, p->copy_stream[(size_t)slot], &w, &h);
    if (rc) return rc;
    if (cudaEventRecord(p->stage_ev[(size_t)b], p->copy_stream[(size_t)slot]) != cudaSuccess) { cudaGetLastError(); return GSEG_E_CUDA; }
    p->stage_next[(size_t)slot] ^= 1;
    pf.input = job->input; pf.bytes = job->jpeg_bytes; pf.w = w; pf.h = h; pf.b = b; pf.valid = true;
    return GSEG_OK;
}

extern "C" int gseg_pool_submit(gseg_pool *p, const gseg_pool_job *job, int64_t *ticket) {
    if (!p || !job || !job->input) return GSEG_E_ARG;
    if (job->out_mode < GSEG_OUT_NONE || job->out_mode > GSEG_OUT_REGIONS) return GSEG_E_ARG;
    if (job->elem_bytes != 0 && job->elem_bytes != 1 && job->elem_bytes != 2 && job->elem_bytes != 4) return GSEG_E_ARG;
    if (job->out_mode != GSEG_OUT_NONE && (!job->out || (job->out_mem_kind != GSEG_MEM_HOST && job->out_mem_kind != GSEG_MEM_DEVICE)))
        return GSEG_E_ARG;
    cudaSetDevice(p->device);
    const int slot = (int)(p->next_ticket % p->S);
    gseg_ctx *c = p->ctx[(size_t)slot];
    // host input: start its copy now, under the kernels of the context's previous job (which reads the other buffer)
    const uint8_t *dev_input = nullptr;
    if (!job->jpeg_bytes && job->mem_kind == GSEG_MEM_HOST && job->w > 0 && job->h > 0 &&
        (size_t)job->w * (size_t)job->h * 3 <= p->stage_bytes) {
        const int b = 2 * slot + p->stage_next[(size_t)slot];
        const size_t row = (size_t)3 * job->w, stride = job->stride_bytes ? (size_t)job->stride_bytes : row;
        cudaError_t e = stage_claim(p, slot, b);
        if (e == cudaSuccess) e = stride == row
                            ? cudaMemcpyAsync(p->stage[(size_t)b], job->input, row * job->h, cudaMemcpyHostToDevice, p->copy_stream[(size_t)slot])
                            : cudaMemcpy2DAsync(p->stage[(size_t)b], row, job->input, stride, row, (size_t)job->h, cudaMemcpyHostToDevice,
                                                p->copy_stream[(size_t)slot]);
        if (e == cudaSuccess) e = cudaEventRecord(p->stage_ev[(size_t)b], p->copy_stream[(size_t)slot]);
        if (e != cudaSuccess) { snprintf(p->err, sizeof(p->err), "submit: input copy: %s", cudaGetErrorString(e)); cudaGetLastError(); return GSEG_E_CUDA; }
        dev_input = p->stage[(size_t)b];
        p->stage_next[(size_t)slot] ^= 1;
    }
    // JPEG input the in-house decoder takes: decoded into the free staging buffer on the copy stream -- already a pipeline
    // turn ago if gseg_pool_run looked ahead, else now (under the last kernels of the context's previous job)
    int jw = 0, jh = 0;
    if (job->jpeg_bytes && job->mem_kind == GSEG_MEM_HOST) {
        gseg_pool::Pref &pf = p->pref[(size_t)slot];
        if (!(pf.valid && pf.input == job->input && pf.bytes == job->jpeg_bytes)) {
            const int drc = jpeg_prefetch(p, slot, job);
            if (drc != GSEG_OK && drc != GSEG_E_UNSUPPORTED && drc != GSEG_E_RANGE) { // not a JPEG at all / CUDA error
                snprintf(p->err, sizeof(p->err), "submit: %s", gseg_last_error(c));
                return drc;
            }
        }
        if (pf.valid) { dev_input = p->stage[(size_t)pf.b]; jw = pf.w; jh = pf.h; pf.valid = false; }
    }
    if (p->busy[(size_t)slot])
        for (Rec &r : p->q)
            if (r.running && r.slot == slot) { retire(p, r); break; }
    Rec r;
    memset(&r, 0, sizeof(r));
    r.job = *job; r.slot = slot; r.running = true; r.ev = nullptr; r.stage_b = -1;
    if (!job->jpeg_bytes && job->mem_kind == GSEG_MEM_DEVICE) { // caller-owned device input (nullptr: the context stages it)
        r.rgb = (const uint8_t *)job->input; r.rgb_stride = job->stride_bytes ? job->stride_bytes : 3 * job->w;
    }
    r.res.ticket = p->next_ticket; r.res.user = job->user; r.res.out = job->out; r.res.w = job->w; r.res.h = job->h;
    int rc;
    if (job->jpeg_bytes && !dev_input) {
        int w = 0, h = 0;
        rc = gseg_segment_jpeg_async(c, job->input, job->jpeg_bytes, &job->params, &w, &h);
        r.res.w = w; r.res.h = h;
    } else if (dev_input) {
        const int b = (int)((dev_input == p->stage[(size_t)(2 * slot)]) ? 2 * slot : 2 * slot + 1);
        const int w = job->jpeg_bytes ? jw : job->w, h = job->jpeg_bytes ? jh : job->h;
        cudaStreamWaitEvent((cudaStream_t)gseg_get_stream(c), p->stage_ev[(size_t)b], 0);
        rc = gseg_segment_async(c, dev_input, w, h, 3 * w, GSEG_MEM_DEVICE, &job->params);
        r.res.w = w; r.res.h = h;
        r.rgb = dev_input; r.rgb_stride = 3 * w; r.stage_b = b;
    } else {
        rc = gseg_segment_async(c, (const uint8_t *)job->input, job->w, job->h, job->stride_bytes ? job->stride_bytes : 3 * job->w,
                                job->mem_kind, &job->params);
    }
    if (rc) { snprintf(p->err, sizeof(p->err), "submit: %s", gseg_last_error(c)); return rc; }
    p->busy[(size_t)slot] = 1;
    p->q.push_back(r);
    if (ticket) *ticket = p->next_ticket;
    ++p->next_ticket;
    return GSEG_OK;
}

extern "C" int gseg_pool_next(gseg_pool *p, gseg_pool_result *out) {
    if (!p || !out) return GSEG_E_ARG;
    if (p->q.empty()) return GSEG_E_STATE;
    cudaSetDevice(p->device);
    Rec &r = p->q.front();
    if (r.running) retire(p, r);
    if (r.ev) {
        if (cudaEventSynchronize(r.ev) != cudaSuccess) { cudaGetLastError(); r.res.status = GSEG_E_CUDA; }
        p->free_ev.push_back(r.ev);
        r.ev = nullptr;
    }
    *out = r.res;
    p->q.pop_front();
    return GSEG_OK;
}

extern "C" int gseg_pool_run(gseg_pool *p, const gseg_pool_job *jobs, int n, gseg_pool_result *results) {
    if (!p || (n > 0 && (!jobs || !results)) || n < 0) return GSEG_E_ARG;
    if (!p->q.empty()) return GSEG_E_STATE; // results of earlier submits would mix in
    for (int sl = 0; sl < p->S; ++sl) { // a look-ahead decode an earlier, failed run left behind must not be mistaken for this run's
        gseg_pool::Pref &pf = p->pref[(size_t)sl];
        if (pf.valid) { p->stage_next[(size_t)sl] = pf.b & 1; pf.valid = false; }
    }
    int first_err = GSEG_OK;
    int got = 0;
    for (int i = 0; i < n; ++i) {
        const int rc = gseg_pool_submit(p, &jobs[i], nullptr);
        if (rc) { first_err = rc; n = i; break; }
        if (i + p->S < n && jobs[i + p->S].jpeg_bytes && jobs[i + p->S].mem_kind == GSEG_MEM_HOST) // the same context's next job
            jpeg_prefetch(p, (int)((p->next_ticket - 1) % p->S), &jobs[i + p->S]);
        // hand finished results out as we go so that the queue stays short
        while ((int)p->q.size() > p->S) { gseg_pool_next(p, &results[got]); ++got; }
    }
    while (got < n) { gseg_pool_next(p, &results[got]); ++got; }
    if (first_err) return first_err;
    for (int i = 0; i < n; ++i)
        if (results[i].status) return results[i].status;
    return GSEG_OK;
}

// The same host<->device copies as a batch (same buffers, same bytes, same round-robin over the contexts' streams),
// no kernels: what the box's PCIe / host memory allows.  `results` = the results of a previous gseg_pool_run of the
// same jobs (they say how many bytes each job sent back).  The jobs' output buffers are overwritten.
extern "C" int gseg_pool_copy_ceiling(gseg_pool *p, const gseg_pool_job *jobs, const gseg_pool_result *results, int n, int reps,
                                      double *ms_per_batch) {
    if (!p || !jobs || !results || n < 1 || reps < 1 || !ms_per_batch) return GSEG_E_ARG;
    if (!p->q.empty()) return GSEG_E_STATE;
    cudaSetDevice(p->device);
    size_t max_in = 0, max_out = 0;
    for (int i = 0; i < n; ++i) {
        const size_t in = jobs[i].jpeg_bytes ? jobs[i].jpeg_bytes : (size_t)3 * jobs[i].w * jobs[i].h;
        if (jobs[i].mem_kind == GSEG_MEM_HOST && in > max_in) max_in = in;
        if (jobs[i].out_mode != GSEG_OUT_NONE && jobs[i].out_mem_kind == GSEG_MEM_HOST && (size_t)results[i].out_bytes > max_out)
            max_out = (size_t)results[i].out_bytes;
    }
    std::vector<void *> din((size_t)p->S, nullptr), dout((size_t)p->S, nullptr);
    std::vector<cudaEvent_t> ends((size_t)p->S, nullptr);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaError_t e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    for (int j = 0; j < p->S && e == cudaSuccess; ++j) {
        if (max_in) e = cudaMalloc(&din[(size_t)j], max_in);
        if (e == cudaSuccess && max_out) e = cudaMalloc(&dout[(size_t)j], max_out);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ends[(size_t)j], cudaEventDisableTiming);
    }
    float ms = 0.f;
    if (e == cudaSuccess) {
        cudaDeviceSynchronize();
        cudaStream_t s0 = (cudaStream_t)gseg_get_stream(p->ctx[0]);
        for (int rep = -1; rep < reps; ++rep) { // rep -1: warm-up
            if (rep == 0) { cudaDeviceSynchronize(); cudaEventRecord(e0, s0); }
            for (int i = 0; i < n; ++i) {
                const int j = i % p->S;
                cudaStream_t s = (cudaStream_t)gseg_get_stream(p->ctx[(size_t)j]);
                const size_t in = jobs[i].jpeg_bytes ? jobs[i].jpeg_bytes : (size_t)3 * jobs[i].w * jobs[i].h;
                if (jobs[i].mem_kind == GSEG_MEM_HOST) cudaMemcpyAsync(din[(size_t)j], jobs[i].input, in, cudaMemcpyHostToDevice, s);
                if (jobs[i].out_mode != GSEG_OUT_NONE && jobs[i].out_mem_kind == GSEG_MEM_HOST && results[i].out_bytes > 0)
                    cudaMemcpyAsync(jobs[i].out, dout[(size_t)j], (size_t)results[i].out_bytes, cudaMemcpyDeviceToHost, s);
            }
        }
        for (int j = 0; j < p->S; ++j) {
            cudaEventRecord(ends[(size_t)j], (cudaStream_t)gseg_get_stream(p->ctx[(size_t)j]));
            cudaStreamWaitEvent(s0, ends[(size_t)j], 0);
        }
        cudaEventRecord(e1, s0);
        e = cudaEventSynchronize(e1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    }
    for (int j = 0; j < p->S; ++j) {
        cudaFree(din[(size_t)j]); cudaFree(dout[(size_t)j]);
        if (ends[(size_t)j]) cudaEventDestroy(ends[(size_t)j]);
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (e != cudaSuccess) { snprintf(p->err, sizeof(p->err), "copy ceiling: %s", cudaGetErrorString(e)); cudaGetLastError(); return GSEG_E_CUDA; }
    *ms_per_batch = (double)ms / reps;
    return GSEG_OK;
}
