// gseg_dedup.cuh -- duplicate-edge elimination between Boruvka rounds (SURVEY.md section 8a row a10).
//
// The reference's DPP branches sort the packed (u', v', w) keys of the contracted graph every round and keep the
// lightest edge of every run of duplicates (Report.pdf p3 s3.2.2 "bit concatenation ... single 64 bit integer";
// p2 s2.2 "only keeping the lightest edge out of all duplicate edges when creating the supervertex").  Here the
// step runs ONCE per image, at the point where it pays (measured, DESIGN.md section 2 item 7): when the graph has
// shrunk to V <= 4096 components while its list still carries E >= 2^19 parallel edges (4K 8-connected hierarchy:
// V = 2.4 k, E = 958 k -> 7 k).  After it the list holds one edge per pair of adjacent components (E ~ 3 V), so every
// remaining round fits the single-cluster tail kernel and touches a handful of pages.  Earlier (V <= 65536) the
// remaining rounds cost less than the sort.
//
//   plan     one block: decide from the device-resident round state; exclusive scan of the page counts
//   keys     pages -> dense arrays: key = (min(a,b) << bits | max(a,b)), payload = dense list position; digit
//            histograms of every pass in the same read
//   sort     the in-house onesweep radix sort (gseg_sort.cuh), device-driven form: ceil(2 bits / 8) passes
//   select   segmented minimum (weight bits, list position) over every run of equal keys, in parallel: runs are
//            reduced by warp shuffles, a run that started in an earlier warp finds its first element with a
//            cooperative 32-ary search, partial minima meet in a 64-bit atomicMin on the run's first element
//   mark     the winner of every run is flagged by its list position; the per-component minima are reset
//   compact  ordered compaction of the flagged edges back into the (now dense) paged list
//   finish   page table + per-component minimum of the next round (seed_dense_pages, as k_graph_init)
//
// Result: unchanged by construction for static weights (FELZ, HIER): the minimum over a set of parallel edges
// is the minimum over the per-pair minima, and the compaction keeps the list order, i.e. the tie-break.  The
// superpixel variant re-weights every edge from the component means each round; fp32 rounding can turn an
// earlier strict order of two parallel edges into a tie that the list position then breaks the other way, so
// its per-pair minimum is not invariant and the step is not run for it.
//
// Every kernel takes its sizes from device memory and exits at once when the plan says "not now": the host
// enqueues the sequence in front of every tail launch without reading anything back.
#pragma once
#include "gseg_sort.cuh"

struct DedupDev {
    SortDev sort;      // sort.active = the plan's decision
    u32 bits;          // bits per component id in the key
    u32 kept;          // edges surviving (written by the compaction)
    u32 tag;           // look-back tag of this invocation's compaction
    u32 seq;           // invocations that ran in this run
    uint2 *xab;        // dense copy of the list: ends
    u32 *xw;           //                          weight bits
    u64 *winner;       // per run (at its first sorted position): min (weight bits << 32 | list position)
    u32 *keep;         // per list position: 1 = survives
    u32 cap;           // capacity of the arrays above, in edges
    u32 min_edges, min_ratio; // run only if E >= min_edges and E >= min_ratio * V
    u32 disabled;
};

__device__ __forceinline__ bool dedup_wanted(const GsegCtl *ctl, const RoundState &st, const DedupDev *dd) {
    return !dd->disabled && !ctl->p.no_dedup && ctl->p.variant != GSEG_SUPERPIX && st.phase != PH_DONE && st.round >= 1u && st.V >= 2u &&
           st.V <= ctl->p.dd_V && st.E <= dd->cap &&
           st.E >= dd->min_edges && st.E / st.V >= dd->min_ratio;
}

__global__ void __launch_bounds__(1024) k_dd_plan(GsegCtl *ctl, GsegBufs B, DedupDev *dd) {
    __shared__ u32 s[34];
    const RoundState st = load_state(ctl);
    const bool go = dedup_wanted(ctl, st, dd);
    if (threadIdx.x == 0) dd->sort.active = go ? 1u : 0u;
    if (!go) return;
    const u32 bits = 32u - (u32)__clz(st.V - 1u); // ids < V fit `bits` bits; V <= 65536 -> key <= 32 bits
    if (threadIdx.x == 0) {
        dd->bits = bits; dd->sort.n = st.E; dd->sort.key_bits = 2u * bits; dd->sort.npass = (2u * bits + 7u) / 8u;
        dd->kept = 0u;
        dd->tag = ctl->p.epoch_base + 2u * GSEG_MAXR + 8u + (dd->seq & 31u);
        dd->seq += 1u;
        ctl->ticketE = 0u;
    }
    for (u32 i = threadIdx.x; i < SORT_MAXPASS * SORT_RADIX; i += blockDim.x) dd->sort.hist[i] = 0u;
    if (threadIdx.x <= SORT_MAXPASS) dd->sort.tickets[threadIdx.x] = 0u;
    block_scan_pages(B.pcnt[st.round & 1], st.P, B.pscan, s);
}

__global__ void __launch_bounds__(NT) k_dd_keys(const GsegCtl *ctl, GsegBufs B, DedupDev *dd) {
    __shared__ u32 sh[SORT_MAXPASS * SORT_RADIX];
    if (!dd->sort.active) return;
    const RoundState st = load_state(ctl);
    const int cur = st.round & 1, lane = threadIdx.x & 31;
    const u32 bits = dd->bits, npass = dd->sort.npass, P = st.P, n = dd->sort.n;
    for (u32 i = threadIdx.x; i < npass * SORT_RADIX; i += NT) sh[i] = 0u;
    // status words of the passes this sort will run
    const size_t nstat = (size_t)npass * ((n + SORT_TILE - 1) / SORT_TILE) * SORT_RADIX;
    for (size_t i = (size_t)blockIdx.x * NT + threadIdx.x; i < nstat; i += (size_t)gridDim.x * NT) dd->sort.status[i] = 0u;
    __syncthreads();
    u64 *keys = dd->sort.keys[0];
    u32 *vals = dd->sort.vals[0];
    for (u32 g = blockIdx.x * (NT / 32) + (threadIdx.x >> 5); g < P; g += gridDim.x * (NT / 32)) {
        const u32 cnt = __ldcg(B.pcnt[cur] + g), src = __ldcg(B.poff[cur] + g), dst = __ldcg(B.pscan + g);
        for (u32 i = lane; i < cnt; i += 32u) {
            const uint2 ab = __ldcg(B.eab[cur] + src + i);
            const u32 w = __ldcg(B.ew[cur] + src + i);
            const u32 key = (min(ab.x, ab.y) << bits) | max(ab.x, ab.y);
            const u32 o = dst + i;
            GSEG_CHK(ctl, o < dd->cap && src + i < ctl->p.edge_slots && ab.x < st.V && ab.y < st.V, 11);
            keys[o] = (u64)key; vals[o] = o;
            dd->xab[o] = ab; dd->xw[o] = w;
            dd->winner[o] = GSEG_KEY_NONE; dd->keep[o] = 0u;
            for (u32 p = 0; p < npass; ++p) atomicAdd(&sh[p * SORT_RADIX + ((key >> (8u * p)) & 255u)], 1u);
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < npass * SORT_RADIX; i += NT)
        if (sh[i]) atomicAdd(&dd->sort.hist[i], sh[i]);
}

// First index of the sorted array whose key equals k, given that index j holds k: 32-ary search by the whole warp
// over [0, j] (all lanes must call; j, k warp-uniform).
__device__ __forceinline__ u32 warp_first_equal(const u64 *__restrict__ K, u32 j, u64 k) {
    const int lane = threadIdx.x & 31;
    u32 lo = 0u, hi = j; // invariant: K[hi] == k, everything below lo is < k
    while (hi > lo) {
        const u32 span = hi - lo, step = (span + 30u) / 31u; // 31 steps cover the span: lane 31 always probes hi
        const u32 probe = min(lo + (u32)lane * step, hi);
        const bool ge = K[probe] >= k; // sorted: true from some lane on
        const u32 m = __ballot_sync(0xFFFFFFFFu, ge);
        const int f = __ffs(m) - 1; // >= 0: K[hi] >= k
        const u32 nhi = min(lo + (u32)f * step, hi);
        const u32 nlo = f > 0 ? min(lo + (u32)(f - 1) * step, hi) + 1u : lo;
        hi = nhi; lo = min(nlo, nhi);
    }
    return hi;
}

// Segmented minimum (weight bits, list position) over every run of equal sorted keys K (payload Vv = list position,
// weights xw by list position); the minimum of a run ends up in winner[first index of the run].
__device__ __forceinline__ void select_runs(const u64 *__restrict__ K, const u32 *__restrict__ Vv, const u32 *__restrict__ xw, u32 n,
                                            u64 *winner) {
    const int lane = threadIdx.x & 31;
    const u32 nr = (n + 31u) & ~31u;
    for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < nr; j += gridDim.x * blockDim.x) {
        const bool act = j < n;
        u64 k = 0;
        u32 v = 0, w = 0xFFFFFFFFu;
        bool head = true;
        if (act) {
            k = K[j]; v = Vv[j]; w = __ldcg(xw + v);
            head = j == 0u || K[j - 1u] != k;
        }
        // runs inside the warp: lane 0 always starts a (partial) run
        const u32 heads = __ballot_sync(0xFFFFFFFFu, head || lane == 0 || !act);
        const u32 above = heads & ~((2u << lane) - 1u);
        const int end = above ? __ffs(above) - 1 : 32;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 ow = __shfl_down_sync(0xFFFFFFFFu, w, o), ov = __shfl_down_sync(0xFFFFFFFFu, v, o);
            if (lane + o < end && (ow < w || (ow == w && ov < v))) { w = ow; v = ov; }
        }
        // where the warp's first run really starts (it may have begun in an earlier warp)
        const u64 k0 = __shfl_sync(0xFFFFFFFFu, k, 0);
        const bool head0 = __shfl_sync(0xFFFFFFFFu, (int)head, 0) != 0;
        const u32 j0 = j - (u32)lane;
        u32 first0 = j0;
        if (!head0 && j0 < n) first0 = warp_first_equal(K, j0, k0);
        if (act && ((heads >> lane) & 1u)) atomicMin(winner + (lane == 0 ? first0 : j), ((u64)w << 32) | (u64)v);
    }
}
__global__ void __launch_bounds__(NT) k_dd_select(DedupDev *dd) {
    if (!dd->sort.active) return;
    const u32 fin = dd->sort.npass & 1u;
    select_runs(dd->sort.keys[fin], dd->sort.vals[fin], dd->xw, dd->sort.n, dd->winner);
}
// Host-sized forms for the export of a strip's graph (gseg_export_graph / gseg_strip_record).
__global__ void __launch_bounds__(NT) k_pair_select_runs(const u64 *__restrict__ K, const u32 *__restrict__ Vv, const u32 *__restrict__ xw,
                                                         u32 n, u64 *winner) {
    select_runs(K, Vv, xw, n, winner);
}
__global__ void __launch_bounds__(NT) k_pair_mark_runs(const u64 *__restrict__ K, const u64 *__restrict__ winner, u32 n, u32 *__restrict__ keep) {
    for (u32 j = blockIdx.x * NT + threadIdx.x; j < n; j += gridDim.x * NT)
        if (j == 0u || K[j - 1u] != K[j]) keep[(u32)__ldcg(winner + j)] = 1u;
}

__global__ void __launch_bounds__(NT) k_dd_mark(const GsegCtl *ctl, GsegBufs B, DedupDev *dd) {
    if (!dd->sort.active) return;
    const RoundState st = load_state(ctl);
    const u32 n = dd->sort.n, fin = dd->sort.npass & 1u;
    const u64 *__restrict__ K = dd->sort.keys[fin];
    for (u32 j = blockIdx.x * NT + threadIdx.x; j < n; j += gridDim.x * NT)
        if (j == 0u || K[j - 1u] != K[j]) dd->keep[(u32)__ldcg(dd->winner + j)] = 1u;
    u64 *best = B.best[st.round & 1];
    for (u32 c = blockIdx.x * NT + threadIdx.x; c < st.V; c += gridDim.x * NT) best[c] = GSEG_KEY_NONE;
}

// Ordered compaction of the flagged edges: chunks of 4 x blockDim list positions by ticket (4 consecutive positions per
// thread), block-granular look-back.
__global__ void __launch_bounds__(1024) k_dd_compact(GsegCtl *ctl, GsegBufs B, DedupDev *dd) {
    __shared__ u32 s[68];
    if (!dd->sort.active) return;
    const RoundState st = load_state(ctl);
    const int cur = st.round & 1, lane = threadIdx.x & 31;
    const u32 CH = 4u * blockDim.x;
    const u32 n = dd->sort.n, nchunks = (n + CH - 1u) / CH, tag = dd->tag;
    for (;;) {
        if (threadIdx.x == 0) s[67] = atomicAdd(&ctl->ticketE, 1u);
        __syncthreads();
        const u32 chunk = s[67];
        if (chunk >= nchunks) break;
        const u32 i0 = chunk * CH + 4u * threadIdx.x;
        u32 kb = 0u;
        if (i0 + 3u < n) {
            const uint4 k4 = *reinterpret_cast<const uint4 *>(dd->keep + i0);
            kb = (k4.x ? 1u : 0u) | (k4.y ? 2u : 0u) | (k4.z ? 4u : 0u) | (k4.w ? 8u : 0u);
        } else {
            for (u32 q = 0; q < 4u; ++q)
                if (i0 + q < n && dd->keep[i0 + q]) kb |= 1u << q;
        }
        const u32 cnt = (u32)__popc(kb);
        const u32 inc = warp_incl_scan(cnt, lane);
        u32 bend;
        const u32 wpre = block_ordered_offset(__shfl_sync(0xFFFFFFFFu, inc, 31), chunk, tag, B.statusE, &ctl->error, s, &bend);
        u32 o = wpre + inc - cnt;
        for (u32 q = 0; q < 4u; ++q)
            if ((kb >> q) & 1u) { B.eab[cur][o] = dd->xab[i0 + q]; B.ew[cur][o] = dd->xw[i0 + q]; ++o; }
        if (chunk == nchunks - 1 && threadIdx.x == 0) dd->kept = bend;
        __syncthreads();
    }
}

// Page table of the dense list and the per-component minimum of the round about to run; the round state takes the new
// edge and page counts.
__global__ void __launch_bounds__(NT) k_dd_finish(GsegCtl *ctl, GsegBufs B, DedupDev *dd) {
    if (!dd->sort.active) return;
    const u32 E = dd->kept, P = (E + GSEG_PAGE - 1u) / GSEG_PAGE;
    // the side as a template argument, and the round state read only where it is needed, keep this kernel at the
    // registers of the seeding loop (32, as k_graph_init)
    if (load_state(ctl).round & 1) seed_dense_pages<1>(B, E, P);
    else seed_dense_pages<0>(B, E, P);
    // the state is read by the kernels AFTER this one; nobody in this kernel reads E or P from it
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&ctl->doneE, 1u) == gridDim.x - 1u) {
            const RoundState st = load_state(ctl);
            ctl->doneE = 0;
            ctl->ticketE = 0; // the compaction's tickets; the next user (k_page_scan) expects zero
            ctl->stDedupIn[st.round] = st.E; ctl->stDedupOut[st.round] = E;
            ctl->st.E = E; ctl->st.P = P;
        }
    }
}
