// gseg_device.cuh -- device-side building blocks shared by every kernel of the engine:
// control block, relaxed global loads/stores, warp/block scans and the single-pass
// decoupled look-back prefix (the scan under every compaction; SURVEY.md section 8a rows a9/a10).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

typedef unsigned int u32;
typedef unsigned long long u64;

#define GSEG_KEY_NONE 0xFFFFFFFFFFFFFFFFull
#define GSEG_INF_BITS 0x7F800000u
#define GSEG_MAXR 64 /* hard cap on rounds per run */
#define GSEG_MAXMASK 64
#define GSEG_PAGE 256u /* slots per page of the edge list = one warp tile (8 rows of 32) */

enum { PH_PRED = 0, PH_MINSIZE = 1, PH_DONE = 2 };
enum { DERR_NONE = 0, DERR_SCAN = 1, DERR_ARENA = 2, DERR_CHASE = 3, DERR_JPEG = 4 /* the in-house JPEG decoder met undecodable data */, DERR_CHECK = 100 /* + site: a bounds check of a checked build */ };

// Checked build (-DGSEG_CHECKED, tools/checked_run.sh): index / capacity assertions at the places where an id, a list slot
// or an arena offset computed on the device is used as an address.  compute-sanitizer is closed on the GPU pool this was
// developed on, so this is the memcheck that could be run: a failed check records its site in the control block and the
// run ends with GSEG_E_INTERNAL.  Compiled out of the product build.
#ifdef GSEG_CHECKED
#define GSEG_CHK(ctl, cond, site)                                                         \
    do {                                                                                  \
        if (!(cond)) atomicMax(&(const_cast<GsegCtl *>(ctl))->error, (u32)DERR_CHECK + (u32)(site)); \
    } while (0)
#else
#define GSEG_CHK(ctl, cond, site) ((void)0)
#endif

// Parameters of one run; filled by the host in pinned memory and copied into GsegCtl::p.
struct GsegRunParams {
    const uint8_t *rgb; // device pointer of the input image (strips: of its first halo row)
    int w, h, stride, D, variant;
    int h_in, y_off;    // strips of a larger image: rows in the input buffer (halo included) and rows of halo above the strip;
                        // the blur reads them instead of clamping at the strip's own edge (whole images: h_in = h, y_off = 0)
    float k;
    int min_size, max_rounds, max_levels;
    u32 arena_cap;  // capacity of the supervertex-map arena in u32 entries
    u32 edge_slots; // capacity of each parity of the edge list, in slots (checked builds)
    u32 epoch_base; // first look-back tag of this run (monotonic across runs)
    int mask_len;
    u32 filter_shift;   // read-before-atomic filter when (E >> filter_shift) > surviving components
    u32 no_dedup;       // GSEG_FLAG_NO_DEDUP: never run the duplicate elimination between rounds
    u32 dd_V;           // ... which runs once the graph has at most this many components (<= 65536: two ids in a 32-bit key)
    u32 tail_E, tail_V, tail_P; // a round with E <= tail_E, V <= tail_V and P <= tail_P runs inside the single-cluster tail kernel
    float mask[GSEG_MAXMASK];
};

// State of the round about to run.  Lives in GsegCtl between kernels of the host-driven schedule
// and in registers inside the persistent round kernel.
struct RoundState { // 8 x u32, read field by field by load_state()
    u32 V, E;      // components / live edges entering the round
    u32 round, phase, levels;
    u32 map_off;   // arena offset of this round's old->new supervertex map
    u32 P;         // pages of the current edge list
    u32 pad;       // (keeps the struct at 8 words)
};

// Device-resident control block: all round-to-round state lives here, so a whole run needs no host
// involvement between rounds (the reference copies a 4-byte flag to the host every round,
// Report.pdf p5).  The host initialises [p .. ticketE] with one H2D copy per run.
struct GsegCtl {
    GsegRunParams p;
    RoundState st;
    u32 Vnext;        // produced by the component scan of the current round
    u32 error;
    u32 ticketC, ticketE; // dynamic tile tickets of the two look-back scans
    u32 doneE;            // blocks that finished the edge phase (the last one advances the round state)
    u32 Eacc[GSEG_MAXR + 1]; // Eacc[r]: edges emitted by round r's edge phase (zeroed by the host; never reset on the device)
    u32 map_skip[GSEG_MAXR + 1]; // 1: round r's map has been folded into an earlier one (arena compaction, FELZ only)
    u32 resume_phase;            // phase the run continues with after the host compacted the arena (error == DERR_ARENA)
    u32 stDedupIn[GSEG_MAXR + 1], stDedupOut[GSEG_MAXR + 1]; // round r ran on a list de-duplicated from In to Out edges (0: no)
    // ---- end of host-initialised head ----
    u32 map_off[GSEG_MAXR + 1];
    u32 stV[GSEG_MAXR], stE[GSEG_MAXR], stM[GSEG_MAXR], stP[GSEG_MAXR], stVafter[GSEG_MAXR];
    u32 stTail[GSEG_MAXR], stPages[GSEG_MAXR]; // 1 when the round ran in the tail kernel; pages of its edge list
    // device timeline (globaltimer, ns): start of the round-0 graph kernel; end of every round; tail rounds
    // also record the ends of their S and R phases and their start
    u64 t_start, t_end[GSEG_MAXR], t_begin[GSEG_MAXR], t_S[GSEG_MAXR], t_R[GSEG_MAXR];
};

// Every device array of a context (both parities of the ping-pong buffers).
struct GsegBufs {
    float *planes, *G, *wgrid;
    u32 *succ, *rank, *wsel, *arena;
    u64 *best[2];     // per component: min outgoing edge key (weight bits << 32 | edge position)
    uint2 *attr[2];   // per component: x = size |C|, y = fp32 bits of Int(C)
    long long *csum[2]; // per component: 3 fixed-point colour sums (superpixel variant)
    float4 *cmean[2];   // per component: mean colour = csum / (256 |C|), computed once per round from the finished sums
    uint2 *eab[2];    // per live edge: the two end components
    u32 *ew[2];       // per live edge: fp32 bits of the weight (superpixel: of the static strength)
    u32 *pcnt[2];     // per page of the edge list: live edges in the page
    u32 *poff[2];     // per page: first slot of the page in eab/ew
    u32 *pscan;       // exclusive scan of pcnt[cur] (re-pack rounds only)
    u64 *statusC, *statusE;
};

__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(u64 *p, u64 v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ u32 ld_relaxed_u32(const u32 *p) {
    u32 v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ u64 globaltimer_ns() {
    u64 t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__device__ __forceinline__ u32 warp_incl_scan(u32 v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// Exclusive scan of one value per thread over a block of NTHR threads. s: >= 34 u32 of shared memory.
// Leaves the block total in s[32]. Contains two __syncthreads().
template <int NTHR>
__device__ __forceinline__ u32 block_excl_scan(u32 v, u32 *s) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    u32 inc = warp_incl_scan(v, lane);
    if (lane == 31) s[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        u32 x = lane < NTHR / 32 ? s[lane] : 0u;
        u32 xi = warp_incl_scan(x, lane);
        s[lane] = xi - x;
        if (lane == 31) s[32] = xi;
    }
    __syncthreads();
    return s[wid] + inc - v;
}

// ---- decoupled look-back ---------------------------------------------------------------------
// status word: [63:34] tag (30 bit, unique per scan launch), [33:32] state, [31:0] value.
#define LB_WIN 4 /* windows of 32 predecessors fetched per look-back round trip */
#define ST_AGG 1u
#define ST_INC 2u
__device__ __forceinline__ u64 pack_status(u32 tag, u32 state, u32 val) {
    return ((u64)((tag << 2) | state) << 32) | (u64)val;
}

// Called by all 32 lanes of warp 0 with the tile's aggregate; returns the exclusive prefix of the
// tile (sum of the aggregates of all lower tiles).  Tiles MUST be handed out through an atomic
// ticket so that every lower tile belongs to a block that is already running.  A bounded spin
// turns a protocol bug into an error code instead of a hung GPU.
// The two halves of the look-back, for callers that can do other work between publishing their aggregate and
// needing their prefix (k_r0_graph resolves a tile after the NEXT tile's stencil work: by then the
// predecessors have published and the walk does not wait).  One warp calls both.
__device__ __forceinline__ void lookback_publish(u64 *status, u32 tile, u32 tag, u32 aggregate) {
    if ((threadIdx.x & 31) == 0) st_relaxed_u64(status + tile, pack_status(tag, tile == 0 ? ST_INC : ST_AGG, aggregate));
}
__device__ __forceinline__ u32 lookback_resolve(u64 *status, u32 tile, u32 tag, u32 aggregate, u32 *err) {
    const int lane = threadIdx.x & 31;
    if (tile == 0) return 0u;
    u32 excl = 0u, spins = 0u;
    int look = (int)tile - 1;
    for (;;) {
        // four windows of 32 predecessors are loaded at once: when a whole generation of tiles starts together
        // nobody has an inclusive prefix yet and every tile has to walk back over all of them, so the walk
        // should cost one round trip per 128 tiles, not per 32
        u64 sv[LB_WIN];
#pragma unroll
        for (int k = 0; k < LB_WIN; ++k) {
            const int idx = look - 32 * k - lane;
            sv[k] = idx >= 0 ? ld_relaxed_u64(status + idx) : pack_status(tag, ST_INC, 0u);
        }
        bool done = false, retry = false;
#pragma unroll
        for (int k = 0; k < LB_WIN; ++k) {
            if (done || retry) break;
            const u32 hi = (u32)(sv[k] >> 32);
            const bool valid = (hi >> 2) == tag && (hi & 3u) != 0u;
            const bool inc = valid && (hi & 3u) == ST_INC;
            const u32 incm = __ballot_sync(0xFFFFFFFFu, inc);
            const u32 invm = __ballot_sync(0xFFFFFFFFu, !valid);
            const int first = incm ? __ffs(incm) - 1 : 32;
            const u32 need = first >= 31 ? 0xFFFFFFFFu : ((2u << first) - 1u);
            if (invm & need) { retry = true; break; } // a predecessor has not published yet: poll again from here
            u32 v = lane <= first ? (u32)sv[k] : 0u;
#pragma unroll
            for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
            excl += v;
            look -= 32;
            if (first < 32) done = true;
        }
        if (done) break;
        if (retry) {
            if (++spins > (1u << 22)) {
                if (lane == 0) *err = DERR_SCAN;
                return excl;
            }
            __nanosleep(spins < 8u ? 100u : 1000u);
        }
    }
    if (lane == 0) st_relaxed_u64(status + tile, pack_status(tag, ST_INC, excl + aggregate));
    return excl;
}
__device__ __forceinline__ u32 lookback_prefix(u64 *status, u32 tile, u32 tag, u32 aggregate, u32 *err) {
    lookback_publish(status, tile, tag, aggregate);
    return lookback_resolve(status, tile, tag, aggregate, err);
}

// Block-granular ordered offsets for warps that each hold one count: the warps of a block exchange
// their counts through shared memory, warp 0 scans them and runs ONE decoupled look-back for the block
// (so the scan has gridDim participants, not gridDim x warps: short look-back walks), and every warp
// gets the global exclusive offset of its items.  Contains two __syncthreads(); sh: >= 66 u32.
// Returns the block's inclusive end (prefix + block total) in *block_end.
__device__ __forceinline__ u32 block_ordered_offset(u32 warp_total, u32 btile, u32 tag, u64 *status, u32 *err, u32 *sh,
                                                    u32 *block_end) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    if (lane == 0) sh[wid] = warp_total;
    __syncthreads();
    if (wid == 0) {
        const u32 v = lane < nwarp ? sh[lane] : 0u;
        const u32 inc = warp_incl_scan(v, lane);
        const u32 tot = __shfl_sync(0xFFFFFFFFu, inc, 31);
        const u32 pre = lookback_prefix(status, btile, tag, tot, err);
        sh[32 + lane] = pre + inc - v;
        if (lane == 0) sh[64] = pre + tot;
    }
    __syncthreads();
    *block_end = sh[64];
    return sh[32 + wid];
}

__device__ __forceinline__ u64 make_key(u32 wbits, u32 idx) { return ((u64)wbits << 32) | (u64)idx; }

// Rows in which no two neighbouring surviving edges share an end on the same side (every run has length one): the shuffle
// minima would reduce nothing.  What such rows do have -- they are the stretches of the list that come from direction-E
// grid edges: a row of the image crosses components A|B|C|..., giving edges (A,B), (B,C), ... -- is that the RIGHT end of
// a surviving edge is the LEFT end of the next surviving one.  So a lane folds the previous surviving lane's key into
// its own before it updates its left end's minimum, and a lane whose right end the next surviving lane takes care of
// issues no second atomic: about one atomic per edge instead of two, 4 shuffles instead of 10.  Valid for any row (the
// equalities are tested, not assumed).  `pos` increases with the lane.  All 32 lanes must call.
__device__ __forceinline__ void warp_chain_min(u64 *best, u32 a, u32 b, u32 kb, u32 pos, bool act, u32 actm) {
    const int lane = threadIdx.x & 31;
    const u32 below = actm & ((1u << lane) - 1u), above = actm & ~((2u << lane) - 1u);
    const int pl = below ? 31 - __clz(below) : lane, nl = above ? __ffs(above) - 1 : lane;
    const u32 pk = __shfl_sync(0xFFFFFFFFu, kb, pl), pp = __shfl_sync(0xFFFFFFFFu, pos, pl), pb = __shfl_sync(0xFFFFFFFFu, b, pl);
    const u32 na = __shfl_sync(0xFFFFFFFFu, a, nl);
#ifndef GSEG_EXP_NOATOMIC
    if (act) {
        u32 ka = kb, qa = pos;
        if (below && pb == a && pk <= kb) { ka = pk; qa = pp; } // the earlier edge wins ties: its position is lower
        atomicMin(best + a, make_key(ka, qa));
        if (!(above && na == b)) atomicMin(best + b, make_key(kb, pos)); // else the next surviving lane folds this edge in
    }
#endif
}

// Segmented min-edge selection (SURVEY.md section 8a row a4) by warp shuffles, both ends of a row of edges at once:
// consecutive lanes that hold edges of the same component form a run; a fixed 5-step segmented min leaves the run's
// minimum key in its first lane, which alone issues the 64-bit atomicMin.  Edge lists are in edge-index order, so a
// component's edges come in long runs (a row segment of a component, a stretch of boundary between two components) and
// the number of atomics falls with the run length.  The two segmented minima (ends ida, idb) are independent dependency
// chains, so interleaving their shuffles halves the latency of the row (these kernels run few warps per SM in late
// rounds and are bound by exactly this chain).
// `pos` MUST increase with the lane index (it is the edge's position in the output list), so among
// equal weights the lower lane already holds the minimum.  All 32 lanes must call.
template <bool FILTER, int WINDOW>
__device__ __forceinline__ void warp_run_min2(u64 *best, u32 ida, u32 idb, u32 kb, u32 pos, bool act, u32 hia, u32 hib,
                                              u32 *sfilter = nullptr) {
    const int lane = threadIdx.x & 31;
    const u32 pa = __shfl_up_sync(0xFFFFFFFFu, ida, 1), pb = __shfl_up_sync(0xFFFFFFFFu, idb, 1);
    const u32 actm = __ballot_sync(0xFFFFFFFFu, act);
    const bool prev_act = lane != 0 && ((actm >> (lane - 1)) & 1u);
    const bool heada = !prev_act || pa != ida, headb = !prev_act || pb != idb;
    const u32 headsa = __ballot_sync(0xFFFFFFFFu, heada || !act), headsb = __ballot_sync(0xFFFFFFFFu, headb || !act);
    if (!FILTER && (headsa & headsb) == 0xFFFFFFFFu) { // warp-uniform: every run has length one on both sides
        warp_chain_min(best, ida, idb, kb, pos, act, actm);
        return;
    }
    if (!act) kb = 0xFFFFFFFFu;
    const u32 hmask = ~((2u << lane) - 1u), lmask = (2u << lane) - 1u;
    const u32 abva = headsa & hmask, abvb = headsb & hmask;
    int enda = abva ? __ffs(abva) - 1 : 32, endb = abvb ? __ffs(abvb) - 1 : 32;
    bool leada = heada, leadb = headb;
    if (WINDOW < 32) {
        // early rounds: runs are short, so reduce inside windows of WINDOW lanes of a run (log2(WINDOW) steps
        // instead of 5) and let every window issue its own atomic
        const int sa = 31 - __clz(headsa & lmask), sb = 31 - __clz(headsb & lmask);
        const int wa = sa + ((lane - sa) & ~(WINDOW - 1)), wb = sb + ((lane - sb) & ~(WINDOW - 1));
        leada = lane == wa; leadb = lane == wb;
        enda = min(enda, wa + WINDOW); endb = min(endb, wb + WINDOW);
    }
    u32 ka = kb, qa = pos, kbb = kb, qb = pos;
#pragma unroll
    for (int o = 1; o < WINDOW; o <<= 1) {
        const u32 oka = __shfl_down_sync(0xFFFFFFFFu, ka, o), oqa = __shfl_down_sync(0xFFFFFFFFu, qa, o);
        const u32 okb = __shfl_down_sync(0xFFFFFFFFu, kbb, o), oqb = __shfl_down_sync(0xFFFFFFFFu, qb, o);
        if (lane + o < enda && oka < ka) { ka = oka; qa = oqa; }
        if (lane + o < endb && okb < kbb) { kbb = okb; qb = oqb; }
    }
    if (FILTER && sfilter) {
        // block-local filter in shared memory (tail, few components): the lightest weight this block has seen
        // per component, seeded from the global minima.  Whoever lowers (or ties) an entry also sends its key
        // to the global minimum, so an entry never promises more than what reaches best[].
        if (leada && act && ka <= atomicMin(sfilter + ida, ka)) atomicMin(best + ida, make_key(ka, qa));
        if (leadb && act && kbb <= atomicMin(sfilter + idb, kbb)) atomicMin(best + idb, make_key(kbb, qb));
        return;
    }
#ifndef GSEG_EXP_NOATOMIC
    // FILTER (components with many edges each): the running minimum only ever decreases, so a key whose weight is
    // above the weight read earlier (hia, hib: the high words of best[ida], best[idb], prefetched for a whole tile at
    // once) can never win; skipping it spares the L2 a same-address atomic
    if (leada && act && (!FILTER || ka <= hia)) atomicMin(best + ida, make_key(ka, qa));
    if (leadb && act && (!FILTER || kbb <= hib)) atomicMin(best + idb, make_key(kbb, qb));
#else
    if (leada && act && ka == 0x12345678u && qa == 77u) best[ida] = make_key(kbb, qb); // keeps the reduction alive
#endif
}

// Same run structure for the size / Int(C) accumulation of phase R: the run's first lane adds the
// run's total size and takes the run's maximum Int.  All 32 lanes must call.
__device__ __forceinline__ void warp_run_accumulate(uint2 *attr, u32 id, u32 sz, u32 iv, bool act) {
    const int lane = threadIdx.x & 31;
    const u32 pid = __shfl_up_sync(0xFFFFFFFFu, id, 1);
    const u32 actm = __ballot_sync(0xFFFFFFFFu, act);
    const bool head = lane == 0 || pid != id || !((actm >> (lane - 1)) & 1u);
    const u32 heads = __ballot_sync(0xFFFFFFFFu, head || !act);
    if (!act) { sz = 0u; iv = 0u; }
    const u32 above = heads & ~((2u << lane) - 1u);
    const int end = above ? __ffs(above) - 1 : 32;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 osz = __shfl_down_sync(0xFFFFFFFFu, sz, o);
        const u32 oiv = __shfl_down_sync(0xFFFFFFFFu, iv, o);
        if (lane + o < end) { sz += osz; iv = max(iv, oiv); }
    }
    if (head && act) {
        atomicAdd(&attr[id].x, sz);
        if (iv) atomicMax(&attr[id].y, iv);
    }
}
