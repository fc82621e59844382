// gseg_regions.cuh -- per-region statistics and region pictures of a finished partition (DESIGN.md section 2 item 10).
//
//   k_regions_init      table records: sums 0, box minimum all ones, box maximum 0
//   k_regions<SMEM>     one pass over the pixels: label (fused map chase, as k_compose / k_compose_px) + input colour,
//                       runs of one label combined in the thread and then across the warp, then
//                         SMEM = true : a block-private table of 32-bit fields in shared memory, flushed with 64-bit
//                                       global atomics (few components)
//                         SMEM = false: 64-bit global atomics straight into the output table (many components)
//   k_region_means      rounded mean colour per component (0xBBGGRR in a u32)
//   k_render<MODE>      mean-colour picture / input with boundaries painted / boundary mask, from a label image
//
// Record of component c (8 x u64): count, sum r, sum g, sum b, sum x, sum y, x0 | y0 << 32, x1 | y1 << 32.  Every word
// is an integer, so the table does not depend on the order of accumulation.  The packed box words are updated as
// four independent 32-bit minima / maxima on their halves (little-endian: x is the low half); one 64-bit min / max
// would order by y first.
#pragma once
#include "gseg_kernels.cuh"

#define RG_K 8       // pixels of one row per thread and step (a chunk never crosses a row)
#define RG_FIELDS 10 // shared-memory record: count, r, g, b, sum x, sum y, x0, y0, x1, y1 (u32, field-major)
#define RG_NONE 0xFFFFFFFFu

#define GSEG_RENDER_MEAN_ 0
#define GSEG_RENDER_OVERLAY_ 1
#define GSEG_RENDER_BOUNDARY_ 2

__global__ void __launch_bounds__(NT) k_regions_init(u64 *__restrict__ table, u32 n) {
    for (u32 c = blockIdx.x * NT + threadIdx.x; c < n; c += gridDim.x * NT) {
        u64 *t = table + 8 * (size_t)c;
#pragma unroll
        for (int k = 0; k < 6; ++k) t[k] = 0ull;
        t[6] = ~0ull;
        t[7] = 0ull;
    }
}

struct RgRun {
    u32 cnt, r, g, b;
    u64 sx, sy;
    u32 x0, y0, x1, y1;
};

template <bool SMEM>
__device__ __forceinline__ void rg_flush(u32 *sm, u32 n, u64 *__restrict__ table, u32 id, const RgRun &a) {
    if (SMEM) { // the pixel bound per block keeps every field below 2^32 (see the launch)
        atomicAdd(&sm[id], a.cnt);
        atomicAdd(&sm[n + id], a.r);
        atomicAdd(&sm[2 * n + id], a.g);
        atomicAdd(&sm[3 * n + id], a.b);
        atomicAdd(&sm[4 * n + id], (u32)a.sx);
        atomicAdd(&sm[5 * n + id], (u32)a.sy);
        atomicMin(&sm[6 * n + id], a.x0);
        atomicMin(&sm[7 * n + id], a.y0);
        atomicMax(&sm[8 * n + id], a.x1);
        atomicMax(&sm[9 * n + id], a.y1);
    } else {
        u64 *t = table + 8 * (size_t)id;
        atomicAdd(&t[0], (u64)a.cnt);
        atomicAdd(&t[1], (u64)a.r);
        atomicAdd(&t[2], (u64)a.g);
        atomicAdd(&t[3], (u64)a.b);
        atomicAdd(&t[4], a.sx);
        atomicAdd(&t[5], a.sy);
        u32 *lo = reinterpret_cast<u32 *>(t + 6), *hi = reinterpret_cast<u32 *>(t + 7);
        atomicMin(&lo[0], a.x0);
        atomicMin(&lo[1], a.y0);
        atomicMax(&hi[0], a.x1);
        atomicMax(&hi[1], a.y1);
    }
}

// Block b takes chunks [b * cpb, min((b + 1) * cpb, nch)); a chunk = RG_K pixels of one row; lane i of a warp takes
// the chunk after lane i-1's, so a uniform region gives every lane one run of the same label.  A thread flushes every
// run that ends inside its chunk (a region boundary: rare for large regions, every few pixels for small ones) and keeps
// its last run open; the open runs of the warp are then combined by label across consecutive lanes (segmented
// shuffle reduction, as warp_run_accumulate) and each segment's first lane flushes once.
template <bool SMEM>
__global__ void __launch_bounds__(NT) k_regions(const GsegCtl *__restrict__ ctl, const u32 *__restrict__ arena, int last,
                                                const u32 *__restrict__ F, const uint8_t *__restrict__ rgb, long long stride,
                                                u32 w, u32 h, u32 n, u32 cpb, u64 *__restrict__ table) {
    extern __shared__ u32 rg_sm[];
    const int lane = threadIdx.x & 31;
    const u32 cpr = (w + RG_K - 1) / RG_K, nch = cpr * h;
    if (SMEM) {
        for (u32 i = threadIdx.x; i < n; i += NT) {
#pragma unroll
            for (int k = 0; k < 6; ++k) rg_sm[k * n + i] = 0u;
            rg_sm[6 * n + i] = RG_NONE; rg_sm[7 * n + i] = RG_NONE;
            rg_sm[8 * n + i] = 0u; rg_sm[9 * n + i] = 0u;
        }
        __syncthreads();
    }
    const u32 begin = blockIdx.x * cpb;
    const u32 end = begin + cpb < nch ? begin + cpb : nch;
    for (u32 base = begin; base < end; base += NT) { // uniform trip count: every lane reaches the shuffles
        const u32 c = base + threadIdx.x;
        const bool act = c < end;
        RgRun a = {0u, 0u, 0u, 0u, 0ull, 0ull, 0u, 0u, 0u, 0u};
        u32 id = RG_NONE;
        if (act) {
            const u32 y = c / cpr, xb = (c - y * cpr) * RG_K;
            const u32 xe = xb + RG_K < w ? xb + RG_K : w;
            const uint8_t *row = rgb + (long long)y * stride;
            // the chunk's RG_K label chases side by side, one map at a time (independent gathers in flight instead of
            // one dependent chain per pixel); pixels past the row's end repeat its last pixel and are not counted
            u32 lab[RG_K];
#pragma unroll
            for (int k = 0; k < RG_K; ++k) lab[k] = arena[y * w + min(xb + (u32)k, xe - 1u)];
            for (int r = 1; r <= last; ++r)
                if (!ctl->map_skip[r]) {
                    const u32 *map = arena + ctl->map_off[r];
#pragma unroll
                    for (int k = 0; k < RG_K; ++k) lab[k] = map[lab[k]];
                }
            if (F) {
#pragma unroll
                for (int k = 0; k < RG_K; ++k) lab[k] = F[lab[k]];
            }
#pragma unroll
            for (int k = 0; k < RG_K; ++k) {
                const u32 x = xb + (u32)k;
                if (x >= xe) break;
                const u32 l = lab[k];
                if (l != id) {
                    if (id != RG_NONE) { a.sy = (u64)y * a.cnt; rg_flush<SMEM>(rg_sm, n, table, id, a); }
                    id = l;
                    a.cnt = a.r = a.g = a.b = 0u; a.sx = 0ull;
                    a.x0 = x; a.y0 = y; a.y1 = y;
                }
                a.cnt += 1u;
                a.r += row[3 * x]; a.g += row[3 * x + 1]; a.b += row[3 * x + 2];
                a.sx += x; a.x1 = x;
            }
            a.sy = (u64)y * a.cnt;
        }
        // combine the open runs of consecutive lanes with the same label
        const u32 pid = __shfl_up_sync(0xFFFFFFFFu, id, 1);
        const u32 actm = __ballot_sync(0xFFFFFFFFu, act);
        const bool head = lane == 0 || pid != id || !((actm >> (lane - 1)) & 1u);
        const u32 heads = __ballot_sync(0xFFFFFFFFu, head || !act);
        const u32 above = heads & ~((2u << lane) - 1u);
        const int send = above ? __ffs(above) - 1 : 32;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 ocnt = __shfl_down_sync(0xFFFFFFFFu, a.cnt, o), orr = __shfl_down_sync(0xFFFFFFFFu, a.r, o);
            const u32 og = __shfl_down_sync(0xFFFFFFFFu, a.g, o), ob = __shfl_down_sync(0xFFFFFFFFu, a.b, o);
            const u64 osx = __shfl_down_sync(0xFFFFFFFFu, a.sx, o), osy = __shfl_down_sync(0xFFFFFFFFu, a.sy, o);
            const u32 ox0 = __shfl_down_sync(0xFFFFFFFFu, a.x0, o), oy0 = __shfl_down_sync(0xFFFFFFFFu, a.y0, o);
            const u32 ox1 = __shfl_down_sync(0xFFFFFFFFu, a.x1, o), oy1 = __shfl_down_sync(0xFFFFFFFFu, a.y1, o);
            if (lane + o < send) {
                a.cnt += ocnt; a.r += orr; a.g += og; a.b += ob; a.sx += osx; a.sy += osy;
                a.x0 = min(a.x0, ox0); a.y0 = min(a.y0, oy0); a.x1 = max(a.x1, ox1); a.y1 = max(a.y1, oy1);
            }
        }
        if (head && act) rg_flush<SMEM>(rg_sm, n, table, id, a);
    }
    if (SMEM) { // flush the block's table: components this block saw
        __syncthreads();
        for (u32 i = threadIdx.x; i < n; i += NT) {
            const u32 cnt = rg_sm[i];
            if (!cnt) continue;
            u64 *t = table + 8 * (size_t)i;
            atomicAdd(&t[0], (u64)cnt);
#pragma unroll
            for (int k = 1; k < 6; ++k) atomicAdd(&t[k], (u64)rg_sm[k * n + i]);
            u32 *lo = reinterpret_cast<u32 *>(t + 6), *hi = reinterpret_cast<u32 *>(t + 7);
            atomicMin(&lo[0], rg_sm[6 * n + i]);
            atomicMin(&lo[1], rg_sm[7 * n + i]);
            atomicMax(&hi[0], rg_sm[8 * n + i]);
            atomicMax(&hi[1], rg_sm[9 * n + i]);
        }
    }
}

// Mean colour of every component, (sum + count / 2) / count per channel (round half up), packed r | g << 8 | b << 16.
__global__ void __launch_bounds__(NT) k_region_means(const u64 *__restrict__ table, u32 n, u32 *__restrict__ mean) {
    for (u32 c = blockIdx.x * NT + threadIdx.x; c < n; c += gridDim.x * NT) {
        const u64 *t = table + 8 * (size_t)c;
        const u64 cnt = t[0], half = cnt >> 1;
        u32 m = 0u;
        if (cnt) m = (u32)((t[1] + half) / cnt) | (u32)((t[2] + half) / cnt) << 8 | (u32)((t[3] + half) / cnt) << 16;
        mean[c] = m;
    }
}

// Boundary pixel: at least one 4-neighbour inside the image has another label (skimage find_boundaries,
// mode="inner", 4-connectivity).
__device__ __forceinline__ bool rg_boundary(const int *__restrict__ labels, u32 p, u32 x, u32 y, u32 w, u32 h, int l) {
    return (x > 0u && labels[p - 1] != l) || (x + 1u < w && labels[p + 1] != l) || (y > 0u && labels[p - w] != l) ||
           (y + 1u < h && labels[p + w] != l);
}

// Four consecutive pixels (row-major, may cross a row) per thread.  MEAN / OVERLAY write 12 bytes: three 32-bit
// stores when the output is 4-byte aligned and the group is whole, else bytes; BOUNDARY writes 4 bytes (one store).
// The input of OVERLAY may have any base alignment and row stride: it is read byte by byte.
template <int MODE>
__global__ void __launch_bounds__(NT) k_render(const int *__restrict__ labels, u32 w, u32 h, const u32 *__restrict__ mean,
                                               const uint8_t *__restrict__ rgb, long long stride, u32 colour,
                                               uint8_t *__restrict__ out, int aligned) {
    const u32 V = w * h, ngroups = (V + 3u) / 4u;
    const uint8_t cr = (uint8_t)(colour >> 16), cgc = (uint8_t)(colour >> 8), cb = (uint8_t)colour;
    for (u32 g = blockIdx.x * NT + threadIdx.x; g < ngroups; g += gridDim.x * NT) {
        const u32 p0 = 4u * g, np = V - p0 < 4u ? V - p0 : 4u;
        uint8_t v[12];
        u32 y = p0 / w, x = p0 - y * w;
#pragma unroll
        for (u32 j = 0; j < 4u; ++j) {
            if (j < np) {
                const u32 p = p0 + j;
                const int l = labels[p];
                if (MODE == GSEG_RENDER_MEAN_) {
                    const u32 m = mean[(u32)l];
                    v[3 * j] = (uint8_t)m; v[3 * j + 1] = (uint8_t)(m >> 8); v[3 * j + 2] = (uint8_t)(m >> 16);
                } else {
                    const bool bd = rg_boundary(labels, p, x, y, w, h, l);
                    if (MODE == GSEG_RENDER_BOUNDARY_) {
                        v[j] = bd ? 1u : 0u;
                    } else if (bd) {
                        v[3 * j] = cr; v[3 * j + 1] = cgc; v[3 * j + 2] = cb;
                    } else {
                        const uint8_t *s = rgb + (long long)y * stride + 3 * (long long)x;
                        v[3 * j] = s[0]; v[3 * j + 1] = s[1]; v[3 * j + 2] = s[2];
                    }
                }
            }
            if (++x == w) { x = 0u; ++y; }
        }
        if (MODE == GSEG_RENDER_BOUNDARY_) {
            if (aligned && np == 4u)
                *reinterpret_cast<u32 *>(out + p0) = (u32)v[0] | (u32)v[1] << 8 | (u32)v[2] << 16 | (u32)v[3] << 24;
            else
#pragma unroll
                for (u32 j = 0; j < 4u; ++j)
                    if (j < np) out[p0 + j] = v[j];
        } else {
            uint8_t *o = out + 3 * (size_t)p0;
            if (aligned && np == 4u) {
                u32 *o4 = reinterpret_cast<u32 *>(o);
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    o4[k] = (u32)v[4 * k] | (u32)v[4 * k + 1] << 8 | (u32)v[4 * k + 2] << 16 | (u32)v[4 * k + 3] << 24;
            } else {
#pragma unroll
                for (u32 j = 0; j < 12u; ++j)
                    if (j < 3u * np) o[j] = v[j];
            }
        }
    }
}
