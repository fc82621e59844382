// gseg_kernels.cuh -- every CUDA kernel of the segmentation hot path (sm_100a).
//
// Stage map (SURVEY.md section 8a):
//   a1  k_blur_tile<R> (k_blur_h/k_blur_v for > 8 taps)  separable Gaussian        Report.pdf p3 s3.2 par.2
//   a2  k_sobel                        Sobel magnitude (superpixel variant)         Report.pdf p4 s3.2.4
//   a3+a4+a6+a7+a9 (round 0)  k_r0_graph: edge weights, min edge per pixel, predicate, 2-cycle
//                                      removal, root renumbering -- one shared-memory tile pass
//                                                                                   Report.pdf p3 s3.2.1, p2-3 s3.1 steps 1,4,5
//   a6+a7+a9 phase_S                   predicate + 2-cycle removal + supervertex renumbering
//   a8  phase_R                        flatten (pointer chase) + size / Int(C) / colour accumulation
//   a10+a4 k_r0_edges, phase_E         edge relabel, self-loop drop, stable compaction, fused with the
//                                      next round's segmented min-edge selection (warp-shuffle run minima)
//   a11 phase_E<SUPERPIX>              per-round re-weighting from component means
//   a12 k_compose*                     hierarchy materialisation                    Report.pdf p4 s3.2.3
//   a13 min-size rounds                phase PH_MINSIZE of phase_S                  Report.pdf p3 step 6
//   a14 k_colorize                     random colour per component                  Report.pdf p4 s3.2.3
//   --  k_tail                         persistent single-cluster kernel: every round whose graph is small
//                                      runs inside one launch with cluster barriers, instead of the
//                                      reference's per-round host loop (Report.pdf p3 "Dynamic
//                                      parallelism", p5 "4 bytes copied back per iteration")
//
// Float contract: every fp32 product, sum, quotient and square root on the weight path is a
// separately rounded IEEE operation (__fmul_rn/__fadd_rn/__fsub_rn/__fdiv_rn/__fsqrt_rn) in the
// order DESIGN.md "Semantics" states; ptxas never contracts these intrinsics into FMAs, so weights
// are bit-identical to the CPU oracle and the total edge order (weight bits, edge index) is too.
#pragma once
#include <cooperative_groups.h>

#include "gseg_device.cuh"

namespace cg = cooperative_groups;

#define NT 256   // threads per block of the grid-wide kernels
#ifndef GSEG_LB_SUCC
#define GSEG_LB_SUCC 4  // resident blocks per SM the successor kernel is compiled for
#endif
#ifndef GSEG_LB_EDGES
#define GSEG_LB_EDGES 4 // ... and the edge kernels (64 registers; more blocks means spills: measured, tools/lb_sweep.sh)
#endif
#define NTT 1024 // threads per block of the single-cluster tail kernel
#define CPT 4    // rows of 32 components per warp tile of phase S
#ifndef RUNWIN
#define RUNWIN 4  // lanes per reduction window of the min-edge selection in rounds without the atomic filter
#endif

// round-0 image tiles
#define TW 64
#ifndef TH
#define TH 32
#endif
#define BW (TW + 4)
#define GH 28            // rows of a round-0 graph tile (28: five 256-thread blocks per SM fit in shared memory)
#define GRPT (GH / 4)    // rows per thread in the successor step: 256 threads = 64 columns x 4 row groups
#define BH (GH + 4)

__constant__ int c_DX[4] = {1, 0, 1, 1};
__constant__ int c_DY[4] = {0, 1, 1, -1};

// Gathers of arrays a PREVIOUS kernel wrote: the grid-wide kernels (one launch per phase) may serve them from
// L1, where neighbouring lanes' lines are already resident; the tail kernel runs every round inside one
// launch, its L1 would hold last round's lines, so it reads through to L2.
template <bool L1, typename T>
__device__ __forceinline__ T ld_prev(const T *p) { return L1 ? *p : __ldcg(p); }

// ------------------------------------------------------------------------------------------------
// a1: separable Gaussian, clamped borders.  u8 interleaved RGB -> 3 fp32 planes.
// Tile kernel: (TW+2R) x (TH+2R) input pixels -> three 8-bit planes in shared memory (32-bit loads of the
// interleaved bytes where the tile is interior and 4-byte aligned, de-interleaved with byte permutes;
// converted to fp32 when the horizontal pass reads them); horizontal pass, shared -> shared (fp32);
// vertical pass -> global.  Each thread produces 8 outputs along the filter direction from 8+2R
// register-held taps (2 shared loads per output instead of 2R+1).  Lanes run ACROSS the filter
// direction (over rows in the horizontal pass, over columns in the vertical pass) and the shared row
// pitches are odd, so every shared access of a warp is bank-conflict free.
// ------------------------------------------------------------------------------------------------
#define BLUR_PF(R) (4 * ((((TW + 2 * (R)) + 3) / 4) | 1)) // byte pitch of the staged input planes: an odd number of words
#define BLUR_PH (TW + 1)                 // pitch of the horizontally filtered planes
template <int R>
__global__ void __launch_bounds__(NT) k_blur_tile(const GsegCtl *__restrict__ ctl, float *__restrict__ planes) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int IW = TW + 2 * R, IH = TH + 2 * R, PF = BLUR_PF(R), PH = BLUR_PH;
    uint8_t *sF = smem_raw;                                      // [3][IH][PF] input planes, still 8-bit (a quarter of
                                                                 // the fp32 staging: five blocks per SM instead of three)
    float *sH = reinterpret_cast<float *>(smem_raw + 3 * IH * PF); // [3][IH][PH] after the horizontal pass
    const int w = ctl->p.w, h = ctl->p.h, stride = ctl->p.stride, h_in = ctl->p.h_in, y_off = ctl->p.y_off;
    const uint8_t *__restrict__ rgb = ctl->p.rgb;
    float m[R + 1];
#pragma unroll
    for (int i = 0; i <= R; ++i) m[i] = ctl->p.mask[i];
    const int ntx = (w + TW - 1) / TW;
    const int x0 = (blockIdx.x % ntx) * TW, y0 = (blockIdx.x / ntx) * TH;
    // 1. stage: 4 pixels (12 interleaved bytes -> one word per colour plane) per item
    const bool fast = x0 - R >= 0 && x0 - R + IW <= w && (stride & 3) == 0 && ((3 * (x0 - R)) & 3) == 0 &&
                      (reinterpret_cast<size_t>(rgb) & 3) == 0 && (IW & 3) == 0;
    constexpr int G4 = (IW + 3) / 4;
    for (int item = threadIdx.x; item < IH * G4; item += NT) {
        const int r = item / G4, g = item - r * G4;
        const int gy = min(max(y0 - R + r + y_off, 0), h_in - 1); // row of the input buffer (halo rows count)
        const uint8_t *row = rgb + (size_t)gy * stride;
        uint8_t *d0 = sF + r * PF + 4 * g;
        if (fast) {
            const uint32_t *wp = reinterpret_cast<const uint32_t *>(row + 3 * (x0 - R) + 12 * g);
            const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2]; // r0 g0 b0 r1 | g1 b1 r2 g2 | b2 r3 g3 b3
            *reinterpret_cast<uint32_t *>(d0) = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);
            *reinterpret_cast<uint32_t *>(d0 + IH * PF) = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);
            *reinterpret_cast<uint32_t *>(d0 + 2 * IH * PF) = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int px = 4 * g + q;
                if (px >= IW) break;
                const int gx = min(max(x0 - R + px, 0), w - 1);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) d0[ch * IH * PF + q] = row[3 * gx + ch];
            }
        }
    }
    __syncthreads();
    // 2. horizontal pass: item = (channel, 8-column group, row); consecutive lanes take consecutive rows
    for (int item = threadIdx.x; item < 3 * (TW / 8) * IH; item += NT) {
        const int r = item % IH, g = (item / IH) % (TW / 8), ch = item / (IH * (TW / 8));
        float v[8 + 2 * R];
        const uint32_t *src = reinterpret_cast<const uint32_t *>(sF + (ch * IH + r) * PF + g * 8);
#pragma unroll
        for (int q = 0; q < (8 + 2 * R + 3) / 4; ++q) {
            const uint32_t t = src[q];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * q + k < 8 + 2 * R) v[4 * q + k] = (float)((t >> (8 * k)) & 255u);
        }
        float *dst = sH + (ch * IH + r) * PH + g * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float s = __fmul_rn(m[0], v[R + j]);
#pragma unroll
            for (int i = 1; i <= R; ++i) s = __fadd_rn(s, __fmul_rn(m[i], __fadd_rn(v[R + j - i], v[R + j + i])));
            dst[j] = s;
        }
    }
    __syncthreads();
    // 3. vertical pass: item = (channel, 8-row group, column); consecutive lanes take consecutive columns
    const u32 V = (u32)w * (u32)h;
    for (int item = threadIdx.x; item < TW * 3 * (TH / 8); item += NT) {
        const int c = item % TW, ch = (item / TW) % 3, rg = item / (3 * TW);
        const int gx = x0 + c;
        if (gx >= w) continue;
        float v[8 + 2 * R];
        const float *src = sH + (ch * IH + rg * 8) * PH + c;
#pragma unroll
        for (int j = 0; j < 8 + 2 * R; ++j) v[j] = src[j * PH];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int gy = y0 + rg * 8 + j;
            if (gy >= h) break;
            float s = __fmul_rn(m[0], v[R + j]);
#pragma unroll
            for (int i = 1; i <= R; ++i) s = __fadd_rn(s, __fmul_rn(m[i], __fadd_rn(v[R + j - i], v[R + j + i])));
            planes[(size_t)ch * V + (size_t)gy * w + gx] = s;
        }
    }
}

// general-sigma fallback (more than 8 one-sided taps)
__global__ void __launch_bounds__(NT) k_blur_h(const GsegCtl *__restrict__ ctl, float *__restrict__ tmp) {
    const int w = ctl->p.w, h = ctl->p.h_in, stride = ctl->p.stride, len = ctl->p.mask_len; // every row of the buffer, halo included
    const uint8_t *__restrict__ rgb = ctl->p.rgb;
    const float *m = ctl->p.mask;
    const u32 V = (u32)w * (u32)h;
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V; p += gridDim.x * NT) {
        const int y = p / w, x = p - y * w;
        const uint8_t *row = rgb + (size_t)y * stride;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float s = __fmul_rn(m[0], (float)row[3 * x + c]);
            for (int i = 1; i < len; ++i) {
                const int xl = max(x - i, 0), xr = min(x + i, w - 1);
                const float pair = __fadd_rn((float)row[3 * xl + c], (float)row[3 * xr + c]);
                s = __fadd_rn(s, __fmul_rn(m[i], pair));
            }
            tmp[(size_t)c * V + p] = s;
        }
    }
}
__global__ void __launch_bounds__(NT) k_blur_v(const GsegCtl *__restrict__ ctl, const float *__restrict__ tmp,
                                               float *__restrict__ planes) {
    const int w = ctl->p.w, h = ctl->p.h, len = ctl->p.mask_len, h_in = ctl->p.h_in, y_off = ctl->p.y_off;
    const float *m = ctl->p.mask;
    const u32 V = (u32)w * (u32)h, Vin = (u32)w * (u32)h_in;
    for (u32 t = blockIdx.x * NT + threadIdx.x; t < 3u * V; t += gridDim.x * NT) {
        const u32 c = t / V, p = t - c * V;
        const int y = p / w + y_off, x = p % w; // y: row in the input buffer
        const float *pl = tmp + (size_t)c * Vin;
        float s = __fmul_rn(m[0], pl[(size_t)y * w + x]);
        for (int i = 1; i < len; ++i) {
            const int yu = max(y - i, 0), yd = min(y + i, h_in - 1);
            const float pair = __fadd_rn(pl[(size_t)yu * w + x], pl[(size_t)yd * w + x]);
            s = __fadd_rn(s, __fmul_rn(m[i], pair));
        }
        planes[t] = s;
    }
}

// a2: Sobel magnitude of the blurred intensity (superpixel variant).
__device__ __forceinline__ float intensity(const float *pl, u32 V, u32 p) {
    return __fmul_rn(__fadd_rn(__fadd_rn(pl[p], pl[V + p]), pl[2 * V + p]), 0.33333334f);
}
__global__ void __launch_bounds__(NT) k_sobel(const GsegCtl *__restrict__ ctl, const float *__restrict__ planes,
                                              float *__restrict__ G) {
    const int w = ctl->p.w, h = ctl->p.h;
    const u32 V = (u32)w * (u32)h;
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V; p += gridDim.x * NT) {
        const int y = p / w, x = p - y * w;
        const int xm = max(x - 1, 0), xp = min(x + 1, w - 1), ym = max(y - 1, 0), yp = min(y + 1, h - 1);
#define AT(xx, yy) intensity(planes, V, (u32)(yy) * w + (xx))
        const float a00 = AT(xm, ym), a10 = AT(x, ym), a20 = AT(xp, ym);
        const float a01 = AT(xm, y), a21 = AT(xp, y);
        const float a02 = AT(xm, yp), a12 = AT(x, yp), a22 = AT(xp, yp);
#undef AT
        const float r = __fadd_rn(__fadd_rn(a20, __fmul_rn(2.0f, a21)), a22);
        const float l = __fadd_rn(__fadd_rn(a00, __fmul_rn(2.0f, a01)), a02);
        const float d = __fadd_rn(__fadd_rn(a02, __fmul_rn(2.0f, a12)), a22);
        const float u = __fadd_rn(__fadd_rn(a00, __fmul_rn(2.0f, a10)), a20);
        const float gx = __fsub_rn(r, l), gy = __fsub_rn(d, u);
        G[p] = __fsqrt_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)));
    }
}

// 24.8 fixed-point colour of a pixel and the superpixel round weight.
__device__ __forceinline__ int fx8(float v) { return __float2int_rn(__fmul_rn(v, 256.0f)); }
__device__ __forceinline__ float mean_dist(const long long *ca, u32 sa, const long long *cb, u32 sb) {
    const float fa = __fmul_rn(__uint2float_rn(sa), 256.0f), fb = __fmul_rn(__uint2float_rn(sb), 256.0f);
    const float dr = __fsub_rn(__fdiv_rn(__ll2float_rn(ca[0]), fa), __fdiv_rn(__ll2float_rn(cb[0]), fb));
    const float dg = __fsub_rn(__fdiv_rn(__ll2float_rn(ca[1]), fa), __fdiv_rn(__ll2float_rn(cb[1]), fb));
    const float db = __fsub_rn(__fdiv_rn(__ll2float_rn(ca[2]), fa), __fdiv_rn(__ll2float_rn(cb[2]), fb));
    const float s = __fadd_rn(__fadd_rn(__fmul_rn(dr, dr), __fmul_rn(dg, dg)), __fmul_rn(db, db));
    return __fsqrt_rn(s);
}

// Superpixel round weight from the per-component means (phase M): the same fp32 operations as mean_dist,
// with the six divisions done once per component instead of once per edge end.
__device__ __forceinline__ float4 mean_of(const long long *csum, const uint2 *attr, u32 n) {
    const float f = __fmul_rn(__uint2float_rn(__ldcg(&attr[n].x)), 256.0f);
    return make_float4(__fdiv_rn(__ll2float_rn(__ldcg(csum + 3 * (size_t)n)), f), __fdiv_rn(__ll2float_rn(__ldcg(csum + 3 * (size_t)n + 1)), f),
                       __fdiv_rn(__ll2float_rn(__ldcg(csum + 3 * (size_t)n + 2)), f), 0.f);
}
__device__ __forceinline__ float mean_dist_m(const float4 *cmean, u32 a, u32 b) {
    const float4 ma = __ldcg(cmean + a), mb = __ldcg(cmean + b);
    const float dr = __fsub_rn(ma.x, mb.x), dg = __fsub_rn(ma.y, mb.y), db = __fsub_rn(ma.z, mb.z);
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dr, dr), __fmul_rn(dg, dg)), __fmul_rn(db, db)));
}

// component-mean distance from the global accumulators (written by atomics in phase R: read at L2)
__device__ __forceinline__ float mean_dist_g(const long long *csum, const uint2 *attr, u32 a, u32 b) {
    long long ca[3] = {__ldcg(csum + 3 * (size_t)a), __ldcg(csum + 3 * (size_t)a + 1), __ldcg(csum + 3 * (size_t)a + 2)};
    long long cb[3] = {__ldcg(csum + 3 * (size_t)b), __ldcg(csum + 3 * (size_t)b + 1), __ldcg(csum + 3 * (size_t)b + 2)};
    return mean_dist(ca, __ldcg(&attr[a].x), cb, __ldcg(&attr[b].x));
}

// Second half of a round-0 graph tile: prefix of the tile's root count (look-back), ids of its roots
// (thread: GRPT rows of one column starting at pixel `pix`, root flags in `flags`, `ex` roots before the
// thread inside the tile) and the cleared accumulators of those ids.
template <bool SP>
__device__ __forceinline__ void r0_finish_tile(GsegCtl *ctl, const GsegBufs &B, u32 tile, u32 total, u32 ex, u32 flags, u32 pix,
                                               u32 tag, u32 ntiles, u32 *s_scan) {
    if (threadIdx.x < 32) {
        const u32 pre = lookback_resolve(B.statusC, tile, tag, total, &ctl->error);
        if (threadIdx.x == 0) s_scan[33] = pre;
    }
    __syncthreads();
    const u32 pre = s_scan[33];
    GSEG_CHK(ctl, (unsigned long long)pre + total <= (unsigned long long)ctl->p.w * ctl->p.h, 1);
    if (tile == ntiles - 1 && threadIdx.x == 0) ctl->Vnext = pre + total;
    const u32 w = (u32)ctl->p.w;
    u32 id = pre + ex;
#pragma unroll
    for (int j = 0; j < GRPT; ++j)
        if (flags & (1u << j)) B.rank[pix + (u32)j * w] = id++;
    // the tile owns the new ids [pre, pre + total): clear their accumulators for phase R / E
    for (u32 i = threadIdx.x; i < total; i += NT) {
        const u32 n = pre + i;
        B.attr[1][n] = make_uint2(0u, 0u); B.best[1][n] = GSEG_KEY_NONE;
        if (SP) { B.csum[1][3 * (size_t)n] = 0; B.csum[1][3 * (size_t)n + 1] = 0; B.csum[1][3 * (size_t)n + 2] = 0; }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// Round 0 on the implicit grid (every pixel is its own component): one tile pass does
//   edge weights (a3) -> per-pixel minimum incident edge (a4; a pure stencil, no atomics) ->
//   predicate (a7) -> 2-cycle removal (a6) -> root flags + look-back scan = new ids (a9).
// Blurred halo: 2 pixels (the 2-cycle test needs the neighbour's choice, which needs the neighbour's
// neighbours).  dir codes: 0..3 own edge (E,S,SE,NE), 4..7 the reverse (W,N,NW,SW); 255 = none.
// Edge index (the tie-break of every comparison) = d*V + p, direction-major.
// New component ids are assigned in tile order (any bijection is valid: ids only name components).
// ------------------------------------------------------------------------------------------------
template <int VARIANT, int D>
__global__ void __launch_bounds__(NT) k_r0_graph(GsegCtl *ctl, GsegBufs B) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr bool SP = VARIANT == GSEG_SUPERPIX;
    float *sP = reinterpret_cast<float *>(smem_raw);   // [3][BH][BW] blurred colour
    float *sW = sP + 3 * BH * BW;                      // [D][BH][BW] own-edge key weights
    float *sG = sW + D * BH * BW;                      // [BH][BW] Sobel (SP only)
    uint8_t *sDir = reinterpret_cast<uint8_t *>(sP);  // [BH-2][BW-2] choices of tile + halo 1; over sP, which is dead after step 2
    __shared__ u32 s_scan[34];
    __shared__ u32 s_tile;
    const int w = ctl->p.w, h = ctl->p.h;
    const u32 V = (u32)w * (u32)h;
    const int ntx = (w + TW - 1) / TW, nty = (h + GH - 1) / GH;
    const u32 ntiles = (u32)ntx * (u32)nty;
    const u32 tag = ctl->p.epoch_base + 1u;
    const float kthr = __fadd_rn(0.0f, __fdiv_rn(ctl->p.k, 1.0f)); // Int = 0, |C| = 1 on both sides
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctl->ticketE = 0; ctl->t_start = globaltimer_ns(); }
    u32 p_tile = 0xFFFFFFFFu, p_total = 0, p_ex = 0, p_flags = 0, p_pix = 0; // the tile whose ids are still to be written
    for (;;) {
        if (threadIdx.x == 0) s_tile = atomicAdd(&ctl->ticketC, 1u);
        __syncthreads();
        const u32 tile = s_tile;
        if (tile >= ntiles) break;
        const int x0 = (int)(tile % ntx) * TW, y0 = (int)(tile / ntx) * GH;
        // 1. blurred halo tile
        for (int i = threadIdx.x; i < BH * BW; i += NT) {
            const int r = i / BW, c = i - r * BW;
            const int gx = x0 - 2 + c, gy = y0 - 2 + r;
            // outside the image: NaN in plane 0 (colour variants), so that every edge touching the pixel
            // gets a NaN weight in step 2 without any bounds test there
            float v0 = SP ? 0.f : __int_as_float(0x7FC00000), v1 = 0.f, v2 = 0.f, g = 0.f;
            if (gx >= 0 && gx < w && gy >= 0 && gy < h) {
                const u32 p = (u32)gy * w + gx;
                v0 = B.planes[p]; v1 = B.planes[V + p]; v2 = B.planes[2 * V + p];
                if (SP) g = B.G[p];
            }
            sP[i] = v0; sP[BH * BW + i] = v1; sP[2 * BH * BW + i] = v2;
            if (SP) sG[i] = g;
        }
        __syncthreads();
        // 2. own-edge weights of every halo-tile pixel (+inf where an end is outside the image).  Edges that
        // leave the halo array read a neighbouring plane / row (always inside shared memory) and produce
        // a value nobody uses: steps 3-4 only read edges with both ends inside the array.
        for (int i = threadIdx.x; i < BH * BW; i += NT) {
            const float p0 = sP[i], p1 = sP[BH * BW + i], p2 = sP[2 * BH * BW + i];
            if (SP) {
                const int r = i / BW, c = i - r * BW;
                const int gx = x0 - 2 + c, gy = y0 - 2 + r;
                const bool in = gx >= 0 && gx < w && gy >= 0 && gy < h;
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const int dx = d == 1 ? 0 : 1, dy = d == 0 ? 0 : (d == 3 ? -1 : 1);
                    const int rr = r + dy, cc = c + dx;
                    float wv = __int_as_float(GSEG_INF_BITS);
                    if (in && rr >= 0 && rr < BH && cc < BW && gx + dx < w && gy + dy < h && gy + dy >= 0) {
                        const int j = rr * BW + cc;
                        long long ca[3] = {fx8(p0), fx8(p1), fx8(p2)};
                        long long cb[3] = {fx8(sP[j]), fx8(sP[BH * BW + j]), fx8(sP[2 * BH * BW + j])};
                        wv = __fmul_rn(__fmul_rn(0.5f, __fadd_rn(sG[i], sG[j])), mean_dist(ca, 1u, cb, 1u));
                    }
                    sW[d * BH * BW + i] = wv;
                }
            } else {
#pragma unroll
                for (int d = 0; d < D; ++d) {
                    const int dx = d == 1 ? 0 : 1, dy = d == 0 ? 0 : (d == 3 ? -1 : 1);
                    const int j = d == 3 ? max(i - BW + 1, 0) : i + dy * BW + dx; // d == 3 from row 0: unused value
                    const float dr = __fsub_rn(p0, sP[j]), dg = __fsub_rn(p1, sP[BH * BW + j]),
                                db = __fsub_rn(p2, sP[2 * BH * BW + j]);
                    const float wv = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dr, dr), __fmul_rn(dg, dg)), __fmul_rn(db, db)));
                    sW[d * BH * BW + i] = wv == wv ? wv : __int_as_float(GSEG_INF_BITS);
                }
            }
        }
        __syncthreads();
        // 3. choice of every pixel of tile + 1-pixel halo: the minimum (weight bits, edge index) over the
        // incident edges.  The edge indices of a pixel's candidates are in a FIXED order (direction-major,
        // then pixel): W < E < N < S < NW < SE < NE < SW  (W, N, NW, SW = the edges owned by the opposite
        // neighbour; for NE the owner of the reverse edge is the pixel below-left, which comes later), so
        // a chain of strict weight comparisons in that order is the key comparison.  Absent edges carry +inf.
        for (int i = threadIdx.x; i < (BH - 2) * (BW - 2); i += NT) {
            const int r = i / (BW - 2) + 1, c = i % (BW - 2) + 1;
            const int gx = x0 - 2 + c, gy = y0 - 2 + r;
            int bdir = 255;
            if (gx >= 0 && gx < w && gy >= 0 && gy < h) {
                const float *w0 = sW + r * BW + c;
                u32 bw = GSEG_INF_BITS, t;
                t = __float_as_uint(w0[-1]);                          if (t < bw) { bw = t; bdir = 4; } // W  (d0 of x-1)
                t = __float_as_uint(w0[0]);                           if (t < bw) { bw = t; bdir = 0; } // E
                t = __float_as_uint(w0[BH * BW - BW]);                if (t < bw) { bw = t; bdir = 5; } // N  (d1 of y-1)
                t = __float_as_uint(w0[BH * BW]);                     if (t < bw) { bw = t; bdir = 1; } // S
                if (D == 4) {
                    t = __float_as_uint(w0[2 * BH * BW - BW - 1]);    if (t < bw) { bw = t; bdir = 6; } // NW (d2 of x-1,y-1)
                    t = __float_as_uint(w0[2 * BH * BW]);             if (t < bw) { bw = t; bdir = 2; } // SE
                    t = __float_as_uint(w0[3 * BH * BW]);             if (t < bw) { bw = t; bdir = 3; } // NE
                    t = __float_as_uint(w0[3 * BH * BW + BW - 1]);    if (t < bw) { bw = t; bdir = 7; } // SW (d3 of x-1,y+1)
                }
                if (VARIANT == GSEG_FELZ && bdir != 255 && !(__uint_as_float(bw) <= kthr)) bdir = 255;
            }
            sDir[(r - 1) * (BW - 2) + (c - 1)] = (uint8_t)bdir;
        }
        __syncthreads();
        // 4. successor (2-cycle removal), outputs, root flags.  Thread: column t%64, rows (t/64)*GRPT + j.
        const int c = (int)(threadIdx.x % TW), rg = (int)(threadIdx.x / TW) * GRPT;
        const int gx = x0 + c;
        u32 flags = 0, cnt = 0;
#pragma unroll
        for (int j = 0; j < GRPT; ++j) {
            const int gy = y0 + rg + j;
            if (gx >= w || gy >= h) continue;
            const u32 p = (u32)gy * w + gx;
            const int r1 = rg + j + 1, c1 = c + 1; // coordinates in sDir
            const int d = sDir[r1 * (BW - 2) + c1];
            u32 s = p, wb = 0;
            if (d != 255) {
                const int dd = d & 3, sgn = d < 4 ? 1 : -1;
                const int dx = sgn * (dd == 1 ? 0 : 1), dy = sgn * (dd == 0 ? 0 : (dd == 3 ? -1 : 1));
                const u32 q = (u32)((int)p + dy * w + dx);
                const int dq = sDir[(r1 + dy) * (BW - 2) + (c1 + dx)];
                s = (dq == (d ^ 4) && p < q) ? p : q;
                // weight of the chosen edge, from its owner's slot
                const int ro = d < 4 ? r1 + 1 : r1 + 1 + dy, co = d < 4 ? c1 + 1 : c1 + 1 + dx;
                wb = __float_as_uint(sW[dd * BH * BW + ro * BW + co]);
            }
            B.succ[p] = s;
            B.wsel[p] = wb;
#pragma unroll
            for (int dd = 0; dd < D; ++dd) {
                float wv = sW[dd * BH * BW + (r1 + 1) * BW + (c1 + 1)];
                if (SP && __float_as_uint(wv) != GSEG_INF_BITS) {
                    const int dx = dd == 1 ? 0 : 1, dy = dd == 0 ? 0 : (dd == 3 ? -1 : 1);
                    wv = __fmul_rn(0.5f, __fadd_rn(sG[(r1 + 1) * BW + c1 + 1], sG[(r1 + 1 + dy) * BW + c1 + 1 + dx]));
                }
                B.wgrid[(size_t)dd * V + p] = wv;
            }
            if (s == p) { flags |= 1u << j; ++cnt; }
        }
        // 5. new ids of the roots, in tile order.  The tile publishes its root count now and takes its
        // prefix one tile later (r0_finish_tile): the look-back of a tile whose predecessors are still in
        // their stencil steps would only wait, so the next tile's stencil runs in that time.
        const u32 ex = block_excl_scan<NT>(cnt, s_scan);
        const u32 total = s_scan[32];
        if (threadIdx.x < 32) lookback_publish(B.statusC, tile, tag, total);
        if (p_tile != 0xFFFFFFFFu) r0_finish_tile<SP>(ctl, B, p_tile, p_total, p_ex, p_flags, p_pix, tag, ntiles, s_scan);
        else __syncthreads(); // s_scan[32] has been read by everybody before the next scan rewrites it
        p_tile = tile; p_total = total; p_ex = ex; p_flags = flags; p_pix = (u32)(y0 + rg) * w + gx;
    }
    if (p_tile != 0xFFFFFFFFu) r0_finish_tile<SP>(ctl, B, p_tile, p_total, p_ex, p_flags, p_pix, tag, ntiles, s_scan);
}

// Round state helpers.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool in_tail(const GsegCtl *ctl, const RoundState &st) {
    return st.round >= 1u && st.E <= ctl->p.tail_E && st.V <= ctl->p.tail_V && st.P <= ctl->p.tail_P;
}

// End-of-round bookkeeping: statistics, phase machine, arena accounting.  Every thread can run it
// redundantly on its private copy of the state; `writer` alone records it in the control block.
__device__ __forceinline__ void advance_state(GsegCtl *ctl, RoundState &st, u32 Vn, u32 En, u32 G, bool writer,
                                              u32 tail_flag = 0u) {
    const u32 r = st.round, V = st.V, merged = V - Vn;
    const int variant = ctl->p.variant;
    u32 phase = st.phase, levels = st.levels;
    if (merged == 0) {
        if (variant == GSEG_FELZ && phase == PH_PRED && ctl->p.min_size > 1) phase = PH_MINSIZE;
        else phase = PH_DONE;
    } else {
        ++levels;
        if (variant != GSEG_FELZ && (Vn <= 1u || (int)levels >= ctl->p.max_levels)) phase = PH_DONE;
    }
    const u32 next_off = st.map_off + V;
    if ((int)(r + 1) >= ctl->p.max_rounds) phase = PH_DONE;
    // The next round's map does not fit the arena: stop here and leave the phase to continue with in the control
    // block.  The host folds the stored maps of a FELZ run into one (only the final partition is needed) and
    // resumes; hierarchy variants at least halve V every round, so their maps always fit.
    bool arena_err = false;
    if (phase != PH_DONE && (u64)next_off + (u64)Vn > (u64)ctl->p.arena_cap) {
        arena_err = true;
        if (writer) ctl->resume_phase = phase;
        phase = PH_DONE;
    }
    if (writer) {
        ctl->stTail[r] = tail_flag; ctl->stPages[r] = st.P;
        ctl->stV[r] = V; ctl->stE[r] = st.E; ctl->stM[r] = merged; ctl->stP[r] = st.phase; ctl->stVafter[r] = Vn;
        ctl->map_off[r] = st.map_off;
        ctl->map_off[r + 1] = next_off;
        ctl->t_end[r] = globaltimer_ns();
        if (arena_err) ctl->error = DERR_ARENA;
    }
    st.P = (st.P + G - 1u) / G; // the edge phase merged G pages into one
    st.round = r + 1; st.levels = levels; st.V = Vn; st.E = En; st.phase = phase; st.map_off = next_off;
    if (writer) ctl->st = st;
}

__device__ __forceinline__ RoundState load_state(const GsegCtl *ctl) {
    RoundState st;
    const u32 *p = reinterpret_cast<const u32 *>(&ctl->st);
    st.V = ld_relaxed_u32(p + 0); st.E = ld_relaxed_u32(p + 1); st.round = ld_relaxed_u32(p + 2); st.phase = ld_relaxed_u32(p + 3);
    st.levels = ld_relaxed_u32(p + 4); st.map_off = ld_relaxed_u32(p + 5); st.P = ld_relaxed_u32(p + 6); st.pad = 0u;
    return st;
}

// Grid-wide kernels: the last block to finish the edge phase advances the round state.  `esum` = this
// block's count of emitted edges (added to the round's total first).
__device__ __forceinline__ void last_block_advance(GsegCtl *ctl, const RoundState &st, u32 G) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&ctl->doneE, 1u) == gridDim.x - 1u) {
            __threadfence();
            ctl->doneE = 0;
            RoundState s2 = st;
            advance_state(ctl, s2, ld_relaxed_u32(&ctl->Vnext), ld_relaxed_u32(&ctl->Eacc[st.round]), G, true);
        }
    }
}

// Pages of the edge list merged into one by this round's edge phase.  Pages start full-ish and lose
// ~45 % of their edges per round; whenever the average page holds fewer than 128 edges the round merges
// G = 2, 4, 8 or 16 consecutive pages into one (so that a merged page receives <= ~256 edges and P keeps
// tracking E / ~150).  The merged pages are written back to back at the offsets of an exclusive scan of
// the INPUT page counts (known before the round starts, so the scan is a tiny separate step, not a
// look-back inside the hot kernel).
__device__ __forceinline__ u32 group_size(const RoundState &st) {
    if (st.P < 2u) return 1u;
    const u32 avg = st.E / st.P; // edges per page entering the round
    if (avg >= 128u) return 1u;
    u32 G = 2u;
    while (G < 16u && (unsigned long long)(2u * G) * avg <= GSEG_PAGE) G *= 2u;
    return G;
}

// Exclusive scan of the page counts by ONE block (any block size that is a multiple of 32, <= 1024), 16
// counts per thread and step (four 16-byte loads in flight: a step costs one memory round trip whatever its
// width).  s: >= 34 u32 of shared memory.  Up to GSEG_PSCAN_INLINE pages this runs as one extra block of the
// successor kernel (and of the tail), beside the work it is independent of; above, k_page_scan does it
// grid-wide.
#define GSEG_PSCAN_INLINE 32768u
#define GSEG_TAIL_STAGE 16384u // components whose map / minima the tail stages in shared memory (2 x 64 KB)
__device__ __forceinline__ void block_scan_pages(const u32 *pcnt, u32 P, u32 *pscan, u32 *s) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    u32 carry = 0;
    for (u32 base = 0; base < P; base += 16u * blockDim.x) {
        const u32 i = base + 16u * threadIdx.x;
        u32 q[16];
        if (i + 15u < P) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint4 t = __ldcg(reinterpret_cast<const uint4 *>(pcnt + i) + k);
                q[4 * k] = t.x; q[4 * k + 1] = t.y; q[4 * k + 2] = t.z; q[4 * k + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) q[k] = i + k < P ? __ldcg(pcnt + i + k) : 0u;
        }
        u32 v = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) { const u32 t = q[k]; q[k] = v; v += t; } // q: exclusive inside the thread
        const u32 inc = warp_incl_scan(v, lane);
        if (lane == 31) s[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const u32 x = lane < nwarp ? s[lane] : 0u;
            const u32 xi = warp_incl_scan(x, lane);
            s[lane] = xi - x;
            if (lane == 31) s[32] = xi;
        }
        __syncthreads();
        const u32 e = carry + s[wid] + inc - v;
        if (i + 15u < P) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                reinterpret_cast<uint4 *>(pscan + i)[k] = make_uint4(e + q[4 * k], e + q[4 * k + 1], e + q[4 * k + 2], e + q[4 * k + 3]);
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k)
                if (i + k < P) pscan[i + k] = e + q[k];
        }
        carry += s[32];
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// a8: flatten + relabel + accumulate.  Chases succ[] to the root (in-place compression is
// race-benign: every value ever stored in a slot is an ancestor of that slot and roots never
// change), maps the component to its root's new id and adds size / Int(C) / colour sums.  Consecutive
// lanes that map to the same new component combine their contributions by warp shuffles first.
// R0: components are pixels (size 1, Int 0, colour = the pixel's fixed-point colour).
// ------------------------------------------------------------------------------------------------
template <int NTH, bool R0, bool SP, bool SPREAD = false>
__device__ __forceinline__ void phase_R(const GsegCtl *ctl, const GsegBufs &B, const RoundState &st) {
    // RPT rows of 32 consecutive components per warp and step: the pointer chases of a thread's RPT components are
    // independent dependency chains, issued together (ncu: the kernel waits on these gathers, 25-28 cycles of
    // long-scoreboard stall per issued instruction with one chain per thread).  Measured on a 2^27-pixel image: rounds
    // >= 1 620 -> 396 us (round 1), 172 -> 111 us (round 2); round 0 (components = pixels, chains short and local,
    // occupancy matters more than chains per thread) 1250 -> 1400 us, so it keeps one chain per thread.
    constexpr int RPT = (SPREAD || R0) ? 1 : 4;
    const int cur = st.round & 1, nxt = cur ^ 1;
    const u32 V = st.V;
    u32 *map = B.arena + st.map_off;
    const u32 V0 = (u32)ctl->p.w * (u32)ctl->p.h;
    const u32 lane = threadIdx.x & 31u, wid = threadIdx.x >> 5, nwarp = NTH / 32;
    // SPREAD (tail): consecutive warps' worth of components go to different blocks (see phase_S)
    const u32 tile0 = SPREAD ? wid * gridDim.x + blockIdx.x : blockIdx.x * nwarp + wid;
    const u32 ntile = (V + 32u * RPT - 1u) / (32u * RPT);
    for (u32 tile = tile0; tile < ntile; tile += gridDim.x * nwarp) {
        u32 c[RPT], r[RPT];
        bool act[RPT], moved[RPT];
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            c[k] = (tile * RPT + (u32)k) * 32u + lane;
            act[k] = c[k] < V;
            r[k] = act[k] ? (SPREAD ? ld_relaxed_u32(B.succ + c[k]) : B.succ[c[k]]) : c[k];
            moved[k] = r[k] != c[k];
        }
        // chase to the roots; stale values are older ancestors: still valid
        bool busy[RPT];
#pragma unroll
        for (int k = 0; k < RPT; ++k) busy[k] = moved[k];
        for (u32 steps = 0;; ++steps) {
            u32 rr[RPT];
            bool any = false;
#pragma unroll
            for (int k = 0; k < RPT; ++k)
                if (busy[k]) rr[k] = SPREAD ? ld_relaxed_u32(B.succ + r[k]) : B.succ[r[k]];
#pragma unroll
            for (int k = 0; k < RPT; ++k)
                if (busy[k]) {
                    if (rr[k] == r[k]) busy[k] = false;
                    else { r[k] = rr[k]; any = true; }
                }
            if (!any) break;
            if (steps > V) { ((GsegCtl *)ctl)->error = DERR_CHASE; break; } // a cycle can only come from a bug: fail, do not hang
        }
        u32 m[RPT], sz[RPT], iv[RPT];
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            m[k] = 0u; sz[k] = 1u; iv[k] = 0u;
            if (act[k]) {
                GSEG_CHK(ctl, r[k] < V, 2);
                if (moved[k]) B.succ[c[k]] = r[k];
                m[k] = ld_prev<!SPREAD>(B.rank + r[k]);
                GSEG_CHK(ctl, m[k] < V && (unsigned long long)st.map_off + c[k] < ctl->p.arena_cap, 3);
            }
        }
#pragma unroll
        for (int k = 0; k < RPT; ++k)
            if (act[k]) {
                map[c[k]] = m[k];
                if (!R0) { const uint2 at = ld_prev<!SPREAD>(B.attr[cur] + c[k]); sz[k] = at.x; iv[k] = at.y; }
                if (moved[k]) iv[k] = max(iv[k], __ldcg(B.wsel + c[k]));
            }
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            warp_run_accumulate(B.attr[nxt], m[k], sz[k], iv[k], act[k]);
            if (SP && act[k]) {
                long long v0, v1, v2;
                const u32 cc = c[k];
                if (R0) { v0 = fx8(B.planes[cc]); v1 = fx8(B.planes[V0 + cc]); v2 = fx8(B.planes[2 * V0 + cc]); }
                else {
                    v0 = __ldcg(B.csum[cur] + 3 * (size_t)cc); v1 = __ldcg(B.csum[cur] + 3 * (size_t)cc + 1);
                    v2 = __ldcg(B.csum[cur] + 3 * (size_t)cc + 2);
                }
                atomicAdd((u64 *)(B.csum[nxt] + 3 * (size_t)m[k]), (u64)v0);
                atomicAdd((u64 *)(B.csum[nxt] + 3 * (size_t)m[k] + 1), (u64)v1);
                atomicAdd((u64 *)(B.csum[nxt] + 3 * (size_t)m[k] + 2), (u64)v2);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Shared tail of the two edge compactions.  A warp tile is ROWS rows of 32 consecutive list entries
// (row j, lane l = entry base + 32 j + l): every load, gather and store of a row touches consecutive
// addresses, and component ids of neighbouring entries are close, so a gather instruction needs a few
// 128-byte lines instead of 32 (the L1 wavefront rate, not HBM, bounds these kernels).  The keep-ballot
// of each row gives every survivor its stable output position without a shuffle scan:
//     pos = tile prefix + survivors in earlier rows + survivors in lower lanes of this row.
// emit_row writes one row's survivors and folds them into the next round's per-component minimum.
// Key = weight bits << 32 | position in the new list (stable compaction keeps list order == edge-index
// order, so position is the same tie-break as the edge index).
// ------------------------------------------------------------------------------------------------
template <bool SP, bool FILTER>
__device__ __forceinline__ void emit_row(const GsegBufs &B, int nxt, u32 pos, bool act, u32 a, u32 b, u32 wv,
                                         u32 fa = 0xFFFFFFFFu, u32 fb = 0xFFFFFFFFu, u32 *sfilter = nullptr) {
    u32 kb = wv;
    if (act) {
#ifndef GSEG_EXP_NOSTORE
        B.eab[nxt][pos] = make_uint2(a, b);
        B.ew[nxt][pos] = wv;
#endif
        if (SP) kb = __float_as_uint(__fmul_rn(__uint_as_float(wv), mean_dist_m(B.cmean[nxt], a, b)));
    }
#ifndef GSEG_EXP_NOMIN
    warp_run_min2<FILTER, FILTER ? 32 : RUNWIN>(B.best[nxt], a, b, kb, pos, act, fa, fb, sfilter);
#endif
}

// Round 0, direction E (pixel p -> p + 1): consecutive lanes are consecutive pixels, so every run of equal ends has length
// one by construction and the row goes straight to the chain form of the minima (warp_chain_min).
template <bool SP>
__device__ __forceinline__ void emit_row_east(const GsegBufs &B, int nxt, u32 pos, bool act, u32 a, u32 b, u32 wv) {
    u32 kb = wv;
    if (act) {
#ifndef GSEG_EXP_NOSTORE
        B.eab[nxt][pos] = make_uint2(a, b);
        B.ew[nxt][pos] = wv;
#endif
        if (SP) kb = __float_as_uint(__fmul_rn(__uint_as_float(wv), mean_dist_m(B.cmean[nxt], a, b)));
    }
#ifndef GSEG_EXP_NOMIN
    warp_chain_min(B.best[nxt], a, b, kb, pos, act, __ballot_sync(0xFFFFFFFFu, act));
#endif
}

// Per-warp bulk copies global -> shared (cp.async.bulk, completion counted in bytes on an mbarrier).
__device__ __forceinline__ u32 smem_addr(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n\tfence.mbarrier_init.release.cluster;" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    asm volatile("{\n\t.reg .pred P1;\n\tWAIT:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
                 "@!P1 bra WAIT;\n\t}" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
// src and dst 16-byte aligned, bytes a non-zero multiple of 16
__device__ __forceinline__ void bulk_copy(void *dst, const void *src, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
// shared memory the warp read with ordinary loads is about to be overwritten by a bulk copy
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Round-0 edge page staging.  A page of direction d reads three streams: map[p] (a ends), map[p + off] (b ends)
// and the weights wgrid[d V + p], p in [p0, min(p0 + 256, V)); only the b stream can start below 0 (NE: off < 0)
// or end past V, and it is clipped to [0, V) (a lane whose b end lies outside is masked anyway).  Each stream is
// copied from the 16-byte boundary at or below its first word to the one at or above its last word: up to 3
// words beyond the live range at each end, inside the allocations (map sits in the arena, which holds >= V + 64
// words; wgrid holds D (V + 64)).
#define R0_STREAM 264                                    // u32 per staged stream: 256 + 2 x 3 alignment words, rounded to 16 B
#define R0_BUF (3 * R0_STREAM)                           // one page: a ends, b ends, weights
#define R0_SMEM ((NT / 32) * (2 * R0_BUF * 4 + 16))      // bytes per block: two page buffers and two mbarriers per warp
struct R0Page {
    int d, off; // direction, pixel offset of the b end
    u32 p0;     // first pixel of the page
    u32 src[3]; // 16-byte aligned first word of each stream: map (a), map (b), wgrid
    u32 n[3];   // words to copy (multiple of 4, may be 0)
};
__device__ __forceinline__ R0Page r0_page(u32 tile, u32 tpd, u32 V, int w) {
    R0Page pg;
    pg.d = (int)(tile / tpd);
    pg.off = pg.d == 0 ? 1 : pg.d == 1 ? w : pg.d == 2 ? w + 1 : 1 - w;
    pg.p0 = (tile - (u32)pg.d * tpd) * GSEG_PAGE;
    const long long end = min((long long)pg.p0 + GSEG_PAGE, (long long)V);
    const long long lo[3] = {pg.p0, max((long long)pg.p0 + pg.off, 0LL), (long long)pg.d * V + pg.p0};
    const long long hi[3] = {end, min(end + pg.off, (long long)V), (long long)pg.d * V + end};
#pragma unroll
    for (int s = 0; s < 3; ++s) {
        pg.src[s] = (u32)(lo[s] & ~3LL);
        pg.n[s] = hi[s] > lo[s] ? (u32)(((hi[s] + 3) & ~3LL) - (lo[s] & ~3LL)) : 0u;
    }
    return pg;
}

// a10 (round 0): grid edges -> paged list of inter-component edges, in edge-index order
// (direction-major: all E edges in pixel order, then S, SE, NE).
//
// PAGED EDGE LIST.  The list is a sequence of pages of GSEG_PAGE = 256 slots; page t holds pcnt[t]
// live edges at slots [256 t, 256 t + pcnt[t]).  List order = page order, then slot order, so the slot
// index of an edge is still a strictly increasing function of its edge index and serves as the
// tie-break.  Compaction is page-local: one warp turns page t of the input into page t of the output
// (8 rows of 32, survivors ranked by row ballots), so the hot kernels need NO global ordered scan, no
// tile tickets, no look-back and no barrier: every warp streams through its pages independently.
// (The decoupled look-back this replaces cost 35-40 % of these kernels: with ~4700 warps starting
// together, each look-back walks back through thousands of not-yet-resolved predecessors.)  Only when
// the pages have become sparse (< 1/4 full) does one round re-pack the list densely with the ordered
// scan; by then the list is small.
//
// STAGED: every page starts with three dependent-free 1 KB reads whose addresses are known long before:
// each warp keeps two page buffers in shared memory and bulk-copies page t + nw into one while it works
// on page t from the other, so the reads of a page overlap the emits of the one before.  Otherwise the
// page's rows are loaded straight into registers (the host picks by pages per warp, R0_STAGE_MAX_PPW).
template <int D, bool SP, bool STAGED>
__global__ void __launch_bounds__(NT, GSEG_LB_EDGES) k_r0_edges(GsegCtl *ctl, GsegBufs B) {
    constexpr int ROWS = GSEG_PAGE / 32;
    extern __shared__ __align__(16) u32 r0_stage[]; // R0_SMEM bytes: [NT / 32][2] mbarriers, then [NT / 32][2][R0_BUF]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const u32 lt = (1u << lane) - 1u;
    const RoundState st = ctl->st; // round 0
    const int w = ctl->p.w, h = ctl->p.h;
    const u32 V = (u32)w * (u32)h;
    const u32 *__restrict__ map = B.arena; // round 0's map sits at arena offset 0
    const u32 *__restrict__ wgrid = reinterpret_cast<const u32 *>(B.wgrid);
    const u32 tpd = (V + GSEG_PAGE - 1) / GSEG_PAGE, ntiles = tpd * (u32)D;
    const u32 nw = gridDim.x * (NT / 32);
    u64 *bar = reinterpret_cast<u64 *>(r0_stage) + 2 * wid;
    u32 *buf = r0_stage + 4 * (NT / 32) + wid * 2 * R0_BUF;
    auto stage = [&](u32 tile, u32 k) { // lane 0: start the copies of page `tile` into buffer k
        const R0Page pg = r0_page(tile, tpd, V, w);
        u32 *dst = buf + k * R0_BUF;
        fence_proxy_async();
        mbar_expect_tx(bar + k, 4u * (pg.n[0] + pg.n[1] + pg.n[2]));
        bulk_copy(dst, map + pg.src[0], 4u * pg.n[0], bar + k); // the a stream is never empty
        if (pg.n[1]) bulk_copy(dst + R0_STREAM, map + pg.src[1], 4u * pg.n[1], bar + k);
        bulk_copy(dst + 2 * R0_STREAM, wgrid + pg.src[2], 4u * pg.n[2], bar + k);
    };
    u32 esum = 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ticketC = 0;
    u32 tile = blockIdx.x * (NT / 32) + wid;
    if constexpr (!STAGED) {
        for (; tile < ntiles; tile += nw) {
            const int d = (int)(tile / tpd);
            const int dx = d == 1 ? 0 : 1, dy = d == 0 ? 0 : (d == 3 ? -1 : 1);
            const int off = dy * w + dx;
            const u32 p0 = (tile - (u32)d * tpd) * GSEG_PAGE + lane;
            u32 a[ROWS], b[ROWS], m[ROWS], wv[ROWS];
            const u32 *wg = wgrid + (size_t)d * V + p0;
            int y = (int)(p0 / (u32)w), x = (int)(p0 - (u32)y * (u32)w);
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
                const u32 p = p0 + 32u * j;
                bool keep = false;
                a[j] = b[j] = wv[j] = 0u;
                if (p < V && x + dx < w && y + dy < h && y + dy >= 0) {
                    a[j] = map[p];
                    b[j] = map[(u32)((int)p + off)];
                    wv[j] = wg[32 * j]; // with the ids, not row by row between the emits: one round trip per page
                    keep = a[j] != b[j];
                }
                m[j] = __ballot_sync(0xFFFFFFFFu, keep);
                x += 32;
                while (x >= w) { x -= w; ++y; }
            }
            u32 total = 0;
#pragma unroll
            for (int j = 0; j < ROWS; ++j) total += __popc(m[j]);
            if (lane == 0) { B.pcnt[1][tile] = total; B.poff[1][tile] = tile * GSEG_PAGE; }
            GSEG_CHK(ctl, (unsigned long long)tile * GSEG_PAGE + total <= ctl->p.edge_slots, 4);
            esum += total;
            u32 rowoff = tile * GSEG_PAGE;
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
                if (m[j] == 0u) continue; // warp-uniform
                const bool act = (m[j] >> lane) & 1u;
                if (d == 0) emit_row_east<SP>(B, 1, rowoff + __popc(m[j] & lt), act, a[j], b[j], wv[j]);
                else emit_row<SP, false>(B, 1, rowoff + __popc(m[j] & lt), act, a[j], b[j], wv[j]);
                rowoff += __popc(m[j]);
            }
        }
    } else {
    if (lane == 0) {
        mbar_init(bar);
        mbar_init(bar + 1);
        if (tile < ntiles) stage(tile, 0u);
    }
    __syncwarp();
    for (u32 it = 0; tile < ntiles; tile += nw, ++it) {
        const u32 k = it & 1u;
        __syncwarp(); // every lane has finished reading buffer k ^ 1 (page tile - nw): refill it
        if (lane == 0 && tile + nw < ntiles) stage(tile + nw, k ^ 1u);
        const R0Page pg = r0_page(tile, tpd, V, w);
        const int d = pg.d, off = pg.off;
        const int dx = d == 1 ? 0 : 1, dy = d == 0 ? 0 : (d == 3 ? -1 : 1);
        const u32 p0 = pg.p0 + lane;
        const u32 *sa = buf + k * R0_BUF + lane;                                          // map[p0 + i]
        const u32 *sb = buf + k * R0_BUF + R0_STREAM + (int)(pg.p0 + off - pg.src[1]) + lane; // map[p0 + off + i]
        const u32 *sw = buf + k * R0_BUF + 2 * R0_STREAM + (d * V + pg.p0 - pg.src[2]) + lane; // wgrid[d V + p0 + i]
        // rows are read from the buffer twice (for the survivor ballots, then for the emits) instead of being
        // held in registers across the emits: 8 rows x (a, b, w) registers less, no spills
        u32 m[ROWS], live = 0u; // live bit j: row j's edge exists (inside the image)
        int y = (int)(p0 / (u32)w), x = (int)(p0 - (u32)y * (u32)w);
        mbar_wait(bar + k, (it >> 1) & 1u);
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
            const u32 p = p0 + 32u * j;
            bool keep = false;
            if (p < V && x + dx < w && y + dy < h && y + dy >= 0) {
                live |= 1u << j;
                keep = sa[32 * j] != sb[32 * j];
            }
            m[j] = __ballot_sync(0xFFFFFFFFu, keep);
            x += 32;
            while (x >= w) { x -= w; ++y; }
        }
        u32 total = 0;
#pragma unroll
        for (int j = 0; j < ROWS; ++j) total += __popc(m[j]);
        if (lane == 0) { B.pcnt[1][tile] = total; B.poff[1][tile] = tile * GSEG_PAGE; }
        GSEG_CHK(ctl, (unsigned long long)tile * GSEG_PAGE + total <= ctl->p.edge_slots, 4);
        esum += total;
        u32 rowoff = tile * GSEG_PAGE;
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
            if (m[j] == 0u) continue; // warp-uniform
            const bool act = (m[j] >> lane) & 1u, in = (live >> j) & 1u;
            const u32 a = in ? sa[32 * j] : 0u, b = in ? sb[32 * j] : 0u, wv = in ? sw[32 * j] : 0u;
            if (d == 0) emit_row_east<SP>(B, 1, rowoff + __popc(m[j] & lt), act, a, b, wv);
            else emit_row<SP, false>(B, 1, rowoff + __popc(m[j] & lt), act, a, b, wv);
            rowoff += __popc(m[j]);
        }
    }
    }
    if (lane == 0 && esum) atomicAdd(&ctl->Eacc[0], esum);
    RoundState s0 = st;
    s0.P = ntiles;
    last_block_advance(ctl, s0, 1u);
}

// ------------------------------------------------------------------------------------------------
// a6+a7+a9 (rounds >= 1): each component's choice under the predicate / min-size rule, 2-cycle
// removal, root flags + look-back scan = new ids; the tile clears the accumulators of its new ids.
// ------------------------------------------------------------------------------------------------
template <bool SP, bool SPREAD>
__device__ __forceinline__ void phase_S(GsegCtl *ctl, const GsegBufs &B, const RoundState &st, u32 *sh) {
    constexpr u32 TILE_C = 32 * CPT; // components per warp: CPT rows of 32 consecutive ids
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const u32 lt = (1u << lane) - 1u;
    const int cur = st.round & 1, nxt = cur ^ 1;
    const u32 V = st.V;
    const u32 nwt = (V + TILE_C - 1) / TILE_C;            // warp tiles
    const u32 ntiles = (nwt + nwarp - 1) / nwarp;         // block tiles = look-back participants
    const u32 tag = ctl->p.epoch_base + st.round * 2u + 1u;
    const u64 *best = B.best[cur];
    const uint2 *eab = B.eab[cur], *attr = B.attr[cur];
    const float kk = ctl->p.k;
    const u32 min_size = (u32)ctl->p.min_size, phase = st.phase;
    const bool pred = ctl->p.variant == GSEG_FELZ && phase == PH_PRED;
    const bool msz = ctl->p.variant == GSEG_FELZ && phase == PH_MINSIZE;
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ticketE = 0;
    // SPREAD (the tail cluster: little work, all blocks resident): warp tiles, statically interleaved over
    // the blocks so that a handful of tiles keeps every SM's issue slots busy instead of one SM's, and a
    // warp-granular look-back.  Otherwise: block tiles by ticket and one look-back per block.
    u32 stile = (u32)wid * gridDim.x + blockIdx.x;
    // ids of a warp tile's roots (row masks m, first id pre) and the cleared accumulators of those ids
    auto write_ids = [&](u32 pre, u32 base, const u32 *m, u32 total) {
        u32 rowoff = pre;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            if ((m[j] >> lane) & 1u) B.rank[base + 32u * j] = rowoff + __popc(m[j] & lt);
            rowoff += __popc(m[j]);
        }
        // the tile owns the new ids [pre, pre + total): clear their accumulators for phase R / E
        for (u32 i = lane; i < total; i += 32u) {
            const u32 n = pre + i;
            B.attr[nxt][n] = make_uint2(0u, 0u); B.best[nxt][n] = GSEG_KEY_NONE;
            if (SP) { B.csum[nxt][3 * (size_t)n] = 0; B.csum[nxt][3 * (size_t)n + 1] = 0; B.csum[nxt][3 * (size_t)n + 2] = 0; }
        }
    };
    // second half of a block tile: prefix of the block's root count, then every warp writes its ids
    auto finish_block = [&](u32 btile, u32 base, u32 below, u32 all, const u32 *m, u32 total) {
        if (wid == 0) {
            const u32 pre = lookback_resolve(B.statusC, btile, tag, all, &ctl->error);
            if (lane == 0) sh[64] = pre;
        }
        __syncthreads();
        const u32 bpre = sh[64];
        if (btile == ntiles - 1 && threadIdx.x == 0) ctl->Vnext = bpre + all;
        write_ids(bpre + below, base, m, total);
        __syncthreads(); // sh[64] is read before the next tile's ticket / prefix overwrite it
    };
    bool p_have = false;
    u32 p_btile = 0, p_base = 0, p_below = 0, p_all = 0, p_total = 0, p_m[CPT] = {};
    for (;;) {
        u32 btile = 0, tile;
        if (SPREAD) {
            tile = stile;
            if (tile >= nwt) break;
            stile += gridDim.x * (u32)nwarp;
        } else {
            if (threadIdx.x == 0) sh[65] = atomicAdd(&ctl->ticketC, 1u);
            __syncthreads();
            btile = sh[65];
            if (btile >= ntiles) break;
            tile = btile * nwarp + wid; // may lie beyond the last warp tile: then every row is empty
        }
        const u32 base = tile * TILE_C + lane;
        // Three dependent gathers per component, each stage issued for all CPT rows at once:
        //   best[c] -> ends of that edge -> {attributes of both ends, best[] of the other end}.
        // The other end s picks c back iff best[s] is this very edge (a lighter edge at s cannot lead to
        // c, or it would be c's minimum too; the predicate is symmetric): that is the 2-cycle test.
        u64 key[CPT], key2[CPT];
        uint2 ab[CPT], ta[CPT], tb[CPT];
#pragma unroll
        for (int j = 0; j < CPT; ++j) key[j] = base + 32u * j < V ? ld_prev<!SPREAD>(best + base + 32u * j) : GSEG_KEY_NONE;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            GSEG_CHK(ctl, key[j] == GSEG_KEY_NONE || (u32)key[j] < ctl->p.edge_slots, 5);
            ab[j] = key[j] != GSEG_KEY_NONE ? ld_prev<!SPREAD>(eab + (u32)key[j]) : make_uint2(0u, 0u);
        }
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            key2[j] = GSEG_KEY_NONE; ta[j] = tb[j] = make_uint2(1u, 0u);
            if (key[j] != GSEG_KEY_NONE) {
                const u32 c = base + 32u * j, other = ab[j].x == c ? ab[j].y : ab[j].x;
                GSEG_CHK(ctl, (ab[j].x == c || ab[j].y == c) && other < V && other != c, 6);
                key2[j] = ld_prev<!SPREAD>(best + other);
                if (pred || msz) { ta[j] = ld_prev<!SPREAD>(attr + ab[j].x); tb[j] = ld_prev<!SPREAD>(attr + ab[j].y); }
            }
        }
        u32 m[CPT], total = 0;
#pragma unroll
        for (int j = 0; j < CPT; ++j) {
            const u32 c = base + 32u * j;
            bool root = false;
            if (c < V) {
                u32 s = c, wb = 0u;
                if (key[j] != GSEG_KEY_NONE) {
                    wb = (u32)(key[j] >> 32);
                    const bool c_is_a = ab[j].x == c;
                    const u32 other = c_is_a ? ab[j].y : ab[j].x;
                    bool ok = true, other_ok = true;
                    if (pred) {
                        const float wt = __uint_as_float(wb);
                        const float fa = __fadd_rn(__uint_as_float(ta[j].y), __fdiv_rn(kk, __uint2float_rn(ta[j].x)));
                        const float fb = __fadd_rn(__uint_as_float(tb[j].y), __fdiv_rn(kk, __uint2float_rn(tb[j].x)));
                        ok = wt <= fa && wt <= fb;
                    } else if (msz) {
                        ok = (c_is_a ? ta[j].x : tb[j].x) < min_size;
                        other_ok = (c_is_a ? tb[j].x : ta[j].x) < min_size;
                    }
                    if (ok) {
                        s = other;
                        if (key2[j] == key[j] && other_ok && c < other) s = c; // 2-cycle: the lower id stays root
                    }
                }
                B.succ[c] = s;
                B.wsel[c] = wb;
                root = s == c;
            }
            m[j] = __ballot_sync(0xFFFFFFFFu, root);
            total += __popc(m[j]);
        }
        if (SPREAD) {
            const u32 pre = lookback_prefix(B.statusC, tile, tag, total, &ctl->error);
            if (tile == nwt - 1 && lane == 0) ctl->Vnext = pre + total;
            write_ids(pre, base, m, total);
        } else {
            // The block publishes its root count now and takes its prefix after the NEXT tile's gathers (see
            // k_r0_graph): a look-back right here mostly waits for predecessors that are still gathering.
            if (lane == 0) sh[wid] = total;
            __syncthreads();
            const u32 v = lane < nwarp ? sh[lane] : 0u;
            u32 below = lane < wid ? v : 0u, all = v;
#pragma unroll
            for (int o = 16; o; o >>= 1) { below += __shfl_xor_sync(0xFFFFFFFFu, below, o); all += __shfl_xor_sync(0xFFFFFFFFu, all, o); }
            if (wid == 0) lookback_publish(B.statusC, btile, tag, all);
            __syncthreads(); // sh[] is free again
            if (p_have) finish_block(p_btile, p_base, p_below, p_all, p_m, p_total);
            p_have = true; p_btile = btile; p_base = base; p_below = below; p_all = all; p_total = total;
#pragma unroll
            for (int j = 0; j < CPT; ++j) p_m[j] = m[j];
        }
    }
    if (!SPREAD && p_have) finish_block(p_btile, p_base, p_below, p_all, p_m, p_total);
}

// ------------------------------------------------------------------------------------------------
// a10 (rounds >= 1): relabel edge ends through this round's map, drop self-loops, page-local stable
// compaction (see k_r0_edges), fused with next round's per-component minimum.  One warp per output
// page = G consecutive input pages read as one virtual page (lanes 0..G-1 hold the counts and offsets
// of the G pages, a 4-step shuffle search maps a virtual slot to its page).  G = 1: page t -> page t in
// place; G > 1: the output page g starts at pscan[G g].  No tickets, no look-back, no barriers.
// ------------------------------------------------------------------------------------------------
template <bool SP, bool SPREAD, int RW>
__device__ __forceinline__ void phase_E_rows(GsegCtl *ctl, const GsegBufs &B, const RoundState &st, u32 Vnext, u32 *stage) {
    constexpr int ROWS = GSEG_PAGE / 32;
    const int lane = threadIdx.x & 31;
    const u32 lt = (1u << lane) - 1u;
    const int cur = st.round & 1, nxt = cur ^ 1;
    const u32 E = st.E, P = st.P;
    const uint2 *eab = B.eab[cur];
    const u32 *ew = B.ew[cur];
    const u32 *pc = B.pcnt[cur], *po = B.poff[cur];
    const u32 *map = B.arena + st.map_off;
    const bool filter = (E >> ctl->p.filter_shift) > Vnext; // many edge ends per surviving component
    const u32 G = group_size(st), ngroups = (P + G - 1u) / G;
    if (blockIdx.x == 0 && threadIdx.x == 0) ctl->ticketC = 0;
    const u32 nwarp = blockDim.x >> 5, nw = gridDim.x * nwarp;
    // Tail with few components: every warp gathers from the same few lines of map[] and best[], and an L2
    // slice serves one request per line at a time (measured: 11 of 16 us of a small round went there).  Each
    // block stages the map and the minima's weights in shared memory once and gathers from there.
    const bool staged = SPREAD && stage != nullptr && st.V <= GSEG_TAIL_STAGE;
    u32 *s_map = stage, *s_bhi = stage + GSEG_TAIL_STAGE;
    if (staged) {
        for (u32 i = threadIdx.x; i < st.V; i += blockDim.x) s_map[i] = __ldcg(map + i);
        if (filter) {
            const u32 *bhi = reinterpret_cast<const u32 *>(B.best[nxt]) + 1;
            for (u32 i = threadIdx.x; i < Vnext; i += blockDim.x) s_bhi[i] = ld_relaxed_u32(bhi + 2 * (size_t)i);
        }
        __syncthreads();
    }
    // RW < 8 (tail rounds with fewer pages than warps): a page is shared by NQ = 8 / RW consecutive warps,
    // RW rows of every 8-row tile each, because a page's latency chain (gathers, then row after row of emits)
    // is what a small round costs.  The warps of a page exchange their survivor counts through shared memory
    // and a named barrier; the slots alternate between tiles, so one barrier per tile is enough.
    constexpr int NQ = ROWS / RW;
    const u32 wid = threadIdx.x >> 5, q = SPREAD ? (wid & (NQ - 1)) : 0u, grp = wid / NQ;
    u32 *s_ex = stage + 2 * GSEG_TAIL_STAGE; // [2][nwarp / NQ][NQ] (SPREAD only)
    u32 esum = 0, parity = 0;
    for (u32 g = SPREAD ? grp * gridDim.x + blockIdx.x : blockIdx.x * nwarp + wid; g < ngroups; g += SPREAD ? gridDim.x * (nwarp / NQ) : nw) {
        u32 mycnt = 0u, myoff = 0u;
        if ((u32)lane < G && G * g + lane < P) { mycnt = __ldcg(pc + G * g + lane); myoff = __ldcg(po + G * g + lane); }
        const u32 incl = warp_incl_scan(mycnt, lane);
        const u32 excl = incl - mycnt, cnt = __shfl_sync(0xFFFFFFFFu, incl, 31);
        const u32 out_base = G > 1u ? __ldcg(B.pscan + G * g) : __shfl_sync(0xFFFFFFFFu, myoff, 0);
        u32 written = 0;
        for (u32 c0 = 0; c0 < cnt; c0 += GSEG_PAGE) { // a virtual page can exceed one 8-row tile
            u32 a[RW], b[RW], wv[RW], m[RW];
#pragma unroll
            for (int j = 0; j < RW; ++j) {
                const u32 i = c0 + 32u * (q * RW + j) + lane;
                u32 k = 0u; // input page of virtual slot i: the last page whose first slot is <= i
                if (G > 1u) {
#pragma unroll
                    for (u32 step = 8u; step; step >>= 1) {
                        const u32 e = __shfl_sync(0xFFFFFFFFu, excl, (int)(k + step));
                        if (k + step < G && e <= i) k += step;
                    }
                }
                const u32 src = __shfl_sync(0xFFFFFFFFu, myoff, (int)k) + (i - __shfl_sync(0xFFFFFFFFu, excl, (int)k));
                uint2 ab = make_uint2(0u, 0u);
                wv[j] = 0u;
                if (i < cnt) {
                    GSEG_CHK(ctl, src < ctl->p.edge_slots, 7);
                    ab = __ldcg(eab + src); wv[j] = __ldcg(ew + src);
                    GSEG_CHK(ctl, ab.x < st.V && ab.y < st.V, 8);
                }
                a[j] = ab.x; b[j] = ab.y;
            }
            u32 sub = 0;
#pragma unroll
            for (int j = 0; j < RW; ++j) {
                bool keep = false;
                if (c0 + 32u * (q * RW + j) + lane < cnt) {
                    if (staged) { a[j] = s_map[a[j]]; b[j] = s_map[b[j]]; }
                    else { a[j] = ld_prev<!SPREAD>(map + a[j]); b[j] = ld_prev<!SPREAD>(map + b[j]); }
                    keep = a[j] != b[j];
                }
                m[j] = __ballot_sync(0xFFFFFFFFu, keep);
                sub += __popc(m[j]);
            }
            u32 before = 0, total = sub; // survivors in the rows of the lower warps of the page / in the whole tile
            if constexpr (NQ > 1) {
                u32 *ex = s_ex + (parity * (nwarp / NQ) + grp) * NQ;
                if (lane == 0) ex[q] = sub;
                asm volatile("bar.sync %0, %1;" ::"r"(1u + grp), "r"(32u * NQ) : "memory");
                total = 0;
#pragma unroll
                for (u32 t = 0; t < (u32)NQ; ++t) { const u32 v = ex[t]; total += v; if (t < q) before += v; }
                parity ^= 1u;
            }
            u32 rowoff = out_base + written + before;
            GSEG_CHK(ctl, (unsigned long long)out_base + written + total <= ctl->p.edge_slots, 9);
            if (filter && staged) {
#pragma unroll
                for (int j = 0; j < RW; ++j) {
                    if (m[j] == 0u) continue; // warp-uniform
                    const bool act = (m[j] >> lane) & 1u;
                    emit_row<SP, true>(B, nxt, rowoff + __popc(m[j] & lt), act, a[j], b[j], wv[j], 0u, 0u, s_bhi);
                    rowoff += __popc(m[j]);
                }
            } else if (filter) {
                // weights of the current minima of both ends, for all rows at once (one round trip)
                u32 fa[RW], fb[RW];
                const u32 *bhi = reinterpret_cast<const u32 *>(B.best[nxt]) + 1; // high word = weight bits
#pragma unroll
                for (int j = 0; j < RW; ++j) {
                    fa[j] = fb[j] = 0xFFFFFFFFu;
                    if ((m[j] >> lane) & 1u) { fa[j] = ld_relaxed_u32(bhi + 2 * (size_t)a[j]); fb[j] = ld_relaxed_u32(bhi + 2 * (size_t)b[j]); }
                }
#pragma unroll
                for (int j = 0; j < RW; ++j) {
                    if (m[j] == 0u) continue; // warp-uniform
                    const bool act = (m[j] >> lane) & 1u;
                    emit_row<SP, true>(B, nxt, rowoff + __popc(m[j] & lt), act, a[j], b[j], wv[j], fa[j], fb[j]);
                    rowoff += __popc(m[j]);
                }
            } else {
#pragma unroll
                for (int j = 0; j < RW; ++j) {
                    if (m[j] == 0u) continue; // warp-uniform
                    const bool act = (m[j] >> lane) & 1u;
                    emit_row<SP, false>(B, nxt, rowoff + __popc(m[j] & lt), act, a[j], b[j], wv[j]);
                    rowoff += __popc(m[j]);
                }
            }
            written += total;
        }
        if (q == 0u) {
            if (lane == 0) { B.pcnt[nxt][g] = written; B.poff[nxt][g] = out_base; }
            esum += written;
        }
    }
    if (lane == 0 && esum) atomicAdd(&ctl->Eacc[st.round], esum);
}
template <bool SP, bool SPREAD = false>
__device__ __forceinline__ void phase_E(GsegCtl *ctl, const GsegBufs &B, const RoundState &st, u32 Vnext, u32 *stage = nullptr) {
    if (SPREAD) {
        const u32 G = group_size(st), ngroups = (st.P + G - 1u) / G;
        // measured on the 16 x 32-warp tail: four warps per page win up to ~2 pages per warp (507 pages: 19.8 ->
        // 13.0 us, 127: 14.4 -> 7.5 us), one warp per page wins beyond (2025 pages: 29.7 vs 35.1 us)
        if (ngroups <= 2u * gridDim.x * (blockDim.x >> 5)) phase_E_rows<SP, true, 2>(ctl, B, st, Vnext, stage);
        else phase_E_rows<SP, true, GSEG_PAGE / 32>(ctl, B, st, Vnext, stage);
    } else {
        phase_E_rows<SP, false, GSEG_PAGE / 32>(ctl, B, st, Vnext, stage);
    }
}

// a11 (superpixel), phase M: mean colour of every component of the next round, from the sums phase R finished.
__device__ __forceinline__ void phase_M(const GsegBufs &B, int nxt, u32 Vnext) {
    for (u32 n = ((threadIdx.x >> 5) * gridDim.x + blockIdx.x) * 32u + (threadIdx.x & 31u); n < Vnext; n += gridDim.x * blockDim.x)
        B.cmean[nxt][n] = mean_of(B.csum[nxt], B.attr[nxt], n); // warps' worth of components interleaved over the blocks
}

// ---- grid-wide schedule: one kernel per phase ---------------------------------------------------
// Every kernel sizes itself from the device-resident round state, so the host enqueues rounds without
// reading anything back; kernels of rounds that are not needed (done / handed to the tail) exit at once.
template <bool R0, bool SP>
__global__ void __launch_bounds__(NT) k_relabel(const GsegCtl *ctl, GsegBufs B) {
    const RoundState st = ctl->st;
    if (st.phase == PH_DONE || in_tail(ctl, st)) return;
    phase_R<NT, R0, SP>(ctl, B, st);
}
__global__ void __launch_bounds__(NT) k_means(const GsegCtl *ctl, GsegBufs B) {
    const RoundState st = ctl->st;
    if (st.phase == PH_DONE || in_tail(ctl, st)) return;
    phase_M(B, (int)((st.round & 1u) ^ 1u), ctl->Vnext);
}
// Merging rounds with more than GSEG_PSCAN_INLINE pages only: the exclusive scan of the page counts the edge
// phase places its output by (smaller ones: block_scan_pages inside k_succ_scan).
// Blocks take chunks of 1024 counts by ticket; chunk prefixes come from a block-granular look-back.
__global__ void __launch_bounds__(1024) k_page_scan(GsegCtl *ctl, GsegBufs B) {
    __shared__ u32 s[68];
    const RoundState st = ctl->st;
    if (st.phase == PH_DONE || in_tail(ctl, st) || group_size(st) == 1u || st.P <= GSEG_PSCAN_INLINE) return;
    const u32 P = st.P, nchunks = (P + 1023u) / 1024u;
    const u32 tag = ctl->p.epoch_base + st.round * 2u + 2u;
    const u32 *pc = B.pcnt[st.round & 1];
    const int lane = threadIdx.x & 31;
    for (;;) {
        if (threadIdx.x == 0) s[67] = atomicAdd(&ctl->ticketE, 1u);
        __syncthreads();
        const u32 chunk = s[67];
        if (chunk >= nchunks) break;
        const u32 i = chunk * 1024u + threadIdx.x;
        const u32 v = i < P ? __ldcg(pc + i) : 0u;
        const u32 inc = warp_incl_scan(v, lane);
        const u32 wtot = __shfl_sync(0xFFFFFFFFu, inc, 31);
        u32 bend;
        const u32 wpre = block_ordered_offset(wtot, chunk, tag, B.statusE, &ctl->error, s, &bend);
        if (i < P) B.pscan[i] = wpre + inc - v;
        __syncthreads();
    }
}
template <bool SP>
__global__ void __launch_bounds__(NT, GSEG_LB_SUCC) k_succ_scan(GsegCtl *ctl, GsegBufs B) {
    __shared__ u32 sh[66];
    const RoundState st = ctl->st;
    if (st.phase == PH_DONE || in_tail(ctl, st)) return;
    if (blockIdx.x == gridDim.x - 1) { // the extra block: page scan of a merging round (block tiles go by ticket, nobody misses it)
        if (group_size(st) > 1u && st.P <= GSEG_PSCAN_INLINE) block_scan_pages(B.pcnt[st.round & 1], st.P, B.pscan, sh);
        return;
    }
    phase_S<SP, false>(ctl, B, st, sh);
}
template <bool SP>
__global__ void __launch_bounds__(NT, GSEG_LB_EDGES) k_edges(GsegCtl *ctl, GsegBufs B) {
    const RoundState st = ctl->st;
    if (st.phase == PH_DONE || in_tail(ctl, st)) return;
    phase_E<SP>(ctl, B, st, ctl->Vnext);
    last_block_advance(ctl, st, group_size(st));
}

// ---- tail schedule: every small round inside one launch of a single thread-block cluster -----------
// Loops S | R | E with three cluster barriers per round until the phase machine says done or the
// graph is (unexpectedly) too large for the tail.  Replaces the reference's host loop with its per-round
// 4-byte read-back and its dynamic-parallelism orchestration kernel (Report.pdf p3, p5).  A cluster is
// co-scheduled by hardware, so tails of different images run side by side on disjoint SMs.
template <bool SP>
__global__ void __launch_bounds__(NTT, 1) k_tail(GsegCtl *ctl, GsegBufs B) {
    extern __shared__ __align__(16) u32 tail_stage[]; // 2 x GSEG_TAIL_STAGE u32 (phase_E)
    __shared__ u32 sh[66];
    cg::cluster_group cl = cg::this_cluster();
    const bool writer = blockIdx.x == 0 && threadIdx.x == 0;
    RoundState st = load_state(ctl);
    cl.sync(); // everyone holds the entry state before the writer may replace it
    while (st.phase != PH_DONE && in_tail(ctl, st)) {
        if (writer) ctl->t_begin[st.round] = globaltimer_ns();
        const u32 G = group_size(st);
        if (G > 1u && blockIdx.x == gridDim.x - 1) block_scan_pages(B.pcnt[st.round & 1], st.P, B.pscan, sh);
        phase_S<SP, true>(ctl, B, st, sh);
        __threadfence();
        cl.sync();
        if (writer) ctl->t_S[st.round] = globaltimer_ns();
        const u32 Vn = ld_relaxed_u32(&ctl->Vnext);
        phase_R<NTT, false, SP, true>(ctl, B, st);
        __threadfence();
        cl.sync();
        if (SP) { // phase M needs the finished sums of phase R and must finish before the edge phase reads the means
            phase_M(B, (int)((st.round & 1u) ^ 1u), Vn);
            __threadfence();
            cl.sync();
        }
        if (writer) ctl->t_R[st.round] = globaltimer_ns();
        phase_E<SP, true>(ctl, B, st, Vn, tail_stage);
        __threadfence();
        cl.sync();
        // One thread advances the round state and publishes it; everybody re-reads it after a fourth
        // barrier.  (Every thread advancing a private copy saves the barrier, but then a thousand copies
        // of the phase machine have to stay bit-identical for the barriers to match up.)
        if (writer) advance_state(ctl, st, Vn, ld_relaxed_u32(&ctl->Eacc[st.round]), G, true, 1u);
        __threadfence();
        cl.sync();
        st = load_state(ctl);
    }
}

// ---- explicit-graph entry (second phase of the tiled schedule) ---------------------------------------
// Export: the live edge list of a finished run, pages gathered into one dense array (one warp per page,
// destination = exclusive scan of the page counts in pscan).
__global__ void __launch_bounds__(1024) k_export_scan(GsegBufs B, int cur, u32 P) {
    __shared__ u32 s[34];
    block_scan_pages(B.pcnt[cur], P, B.pscan, s);
}
__global__ void __launch_bounds__(NT) k_export_gather(GsegBufs B, int cur, u32 P) {
    const int lane = threadIdx.x & 31;
    const int nxt = cur ^ 1;
    for (u32 g = blockIdx.x * (NT / 32) + (threadIdx.x >> 5); g < P; g += gridDim.x * (NT / 32)) {
        const u32 cnt = B.pcnt[cur][g], src = B.poff[cur][g], dst = B.pscan[g];
        for (u32 i = lane; i < cnt; i += 32u) { B.eab[nxt][dst + i] = B.eab[cur][src + i]; B.ew[nxt][dst + i] = B.ew[cur][src + i]; }
    }
}
// Duplicate elimination of the exported list (the reference's DPP branches: sort packed keys, keep the
// lightest of every run, Report.pdf p3 s3.2.2): key = pair of end components, payload = list position;
// after the in-house onesweep sort the minimum (weight bits, position) of every run is found in parallel
// (k_pair_select_runs / k_pair_mark_runs, gseg_dedup.cuh) and that edge is marked; the marked edges are compacted in
// list order.
__global__ void __launch_bounds__(NT) k_pair_keys(const uint2 *__restrict__ eab, u32 E, u32 V, u64 *__restrict__ keys,
                                                  u32 *__restrict__ vals, u32 *__restrict__ keep) {
    for (u32 i = blockIdx.x * NT + threadIdx.x; i < E; i += gridDim.x * NT) {
        const uint2 ab = eab[i];
        keys[i] = (u64)min(ab.x, ab.y) * V + max(ab.x, ab.y);
        vals[i] = i;
        keep[i] = 0u;
    }
}
// Ordered compaction of the marked edges: chunks of blockDim edges by ticket, block-granular look-back.
__global__ void __launch_bounds__(1024) k_compact_keep(GsegCtl *ctl, const uint2 *__restrict__ eab, const u32 *__restrict__ ew,
                                                       const u32 *__restrict__ keep, u32 E, u32 tag, u64 *status,
                                                       uint2 *__restrict__ oab, u32 *__restrict__ ow) {
    __shared__ u32 s[68];
    const int lane = threadIdx.x & 31;
    const u32 nchunks = (E + blockDim.x - 1) / blockDim.x;
    for (;;) {
        if (threadIdx.x == 0) s[67] = atomicAdd(&ctl->ticketE, 1u);
        __syncthreads();
        const u32 chunk = s[67];
        if (chunk >= nchunks) break;
        const u32 i = chunk * blockDim.x + threadIdx.x;
        const bool k = i < E && keep[i] != 0u;
        const u32 m = __ballot_sync(0xFFFFFFFFu, k);
        u32 bend;
        const u32 wpre = block_ordered_offset(__popc(m), chunk, tag, status, &ctl->error, s, &bend);
        if (k) { const u32 o = wpre + __popc(m & ((1u << lane) - 1u)); oab[o] = eab[i]; ow[o] = ew[i]; }
        if (chunk == nchunks - 1 && threadIdx.x == 0) ctl->Eacc[GSEG_MAXR] = bend;
        __syncthreads();
    }
}
// Import: dense pages of GSEG_PAGE slots over a caller-supplied edge list (slot = list position = the
// tie-break) and the per-component minimum of round 1.
__global__ void __launch_bounds__(NT) k_graph_init(GsegBufs B, u32 E, u32 P) {
    const int lane = threadIdx.x & 31;
    for (u32 g = blockIdx.x * (NT / 32) + (threadIdx.x >> 5); g < P; g += gridDim.x * (NT / 32)) {
        if (lane == 0) { B.pcnt[1][g] = min(GSEG_PAGE, E - g * GSEG_PAGE); B.poff[1][g] = g * GSEG_PAGE; }
#pragma unroll
        for (int j = 0; j < (int)(GSEG_PAGE / 32); ++j) {
            const u32 e = g * GSEG_PAGE + 32u * j + lane;
            const bool act = e < E;
            uint2 ab = make_uint2(0u, 0u);
            u32 wv = 0u;
            if (act) { ab = B.eab[1][e]; wv = B.ew[1][e]; }
            warp_run_min<false, 32>(B.best[1], ab.x, wv, e, act, 0xFFFFFFFFu);
            warp_run_min<false, 32>(B.best[1], ab.y, wv, e, act, 0xFFFFFFFFu);
        }
    }
}

// ---- tiled schedule on the device (BASELINE.json configs[4]; DESIGN.md "Tiled schedule") ---------------
// Strip record (32-bit words, device memory): header[8] = {magic, nV, nE, w, 0...} | attr uint2[nV] (size, Int bits)
// | eab uint2[nE] | ew u32[nE] | top_lab[w] | bot_lab[w] | top_col f32[3][w] | bot_col f32[3][w].
#define GSEG_REC_MAGIC 0x47534731u
#define GSEG_REC_HEAD 8u
#define GSEG_MAX_STRIPS 64
__host__ __device__ __forceinline__ size_t rec_words(size_t nV, size_t nE, size_t w) { return GSEG_REC_HEAD + 2 * nV + 3 * nE + 8 * w; }

// header + first / last row of the strip's dense label image and of its blurred planes
__global__ void __launch_bounds__(NT) k_record_rows(const int *__restrict__ labels, const float *__restrict__ planes, u32 w, u32 h,
                                                    u32 nV, u32 nE, u32 *__restrict__ rec) {
    const size_t V = (size_t)w * h;
    u32 *top_lab = rec + GSEG_REC_HEAD + 2 * (size_t)nV + 3 * (size_t)nE, *bot_lab = top_lab + w;
    float *top_col = reinterpret_cast<float *>(bot_lab + w), *bot_col = top_col + 3 * (size_t)w;
    if (blockIdx.x == 0 && threadIdx.x < GSEG_REC_HEAD)
        rec[threadIdx.x] = threadIdx.x == 0 ? GSEG_REC_MAGIC : threadIdx.x == 1 ? nV : threadIdx.x == 2 ? nE : threadIdx.x == 3 ? w : 0u;
    for (u32 x = blockIdx.x * NT + threadIdx.x; x < w; x += gridDim.x * NT) {
        top_lab[x] = (u32)labels[x];
        bot_lab[x] = (u32)labels[(size_t)(h - 1) * w + x];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            top_col[(size_t)c * w + x] = planes[c * V + x];
            bot_col[(size_t)c * w + x] = planes[c * V + (size_t)(h - 1) * w + x];
        }
    }
}

struct JoinDesc {
    u32 n_strips, w, conn, ncut; // ncut: cut edges per strip boundary (w, or w + 2 (w - 1) when 8-connected)
    unsigned long long stride_words;   // distance between the gathered records
    u32 voff[GSEG_MAX_STRIPS + 1];     // first joined component id of strip s
    u32 ne[GSEG_MAX_STRIPS];           // edges of strip s
    u32 eoff[GSEG_MAX_STRIPS + 1];     // list position of strip s's first own edge; its cut edges to s + 1 follow them
};
__device__ __forceinline__ float l2_rn(float a0, float a1, float a2, float b0, float b1, float b2) {
    const float dr = __fsub_rn(a0, b0), dg = __fsub_rn(a1, b1), db = __fsub_rn(a2, b2);
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dr, dr), __fmul_rn(dg, dg)), __fmul_rn(db, db)));
}
// The join on the device: components renumbered strip by strip (id + voff[s]); list = strip 0's edges, the cut
// edges 0|1 (S for x = 0..w-1, then SE, then NE; weight = L2 distance of the two blurred end pixels, same
// operation order as k_r0_graph), strip 1's edges, ...  Writes the graph where k_graph_init expects it.
__global__ void __launch_bounds__(NT) k_join(const __grid_constant__ JoinDesc jd, const u32 *__restrict__ recs, GsegBufs B) {
    const u32 S = jd.n_strips, w = jd.w;
    const u32 Vtot = jd.voff[S], Etot = jd.eoff[S];
    for (size_t i = (size_t)blockIdx.x * NT + threadIdx.x; i < (size_t)Vtot + Etot; i += (size_t)gridDim.x * NT) {
        if (i < Vtot) {
            u32 s = 0;
            while (s + 1 < S && jd.voff[s + 1] <= (u32)i) ++s;
            const u32 *rec = recs + (size_t)s * jd.stride_words;
            B.attr[1][i] = reinterpret_cast<const uint2 *>(rec + GSEG_REC_HEAD)[(u32)i - jd.voff[s]];
            B.best[1][i] = GSEG_KEY_NONE;
            continue;
        }
        const u32 j = (u32)(i - Vtot);
        u32 s = 0;
        while (s + 1 < S && jd.eoff[s + 1] <= j) ++s;
        const u32 *rec = recs + (size_t)s * jd.stride_words;
        const u32 nV = jd.voff[s + 1] - jd.voff[s], nE = jd.ne[s], k = j - jd.eoff[s];
        if (k < nE) { // one of the strip's own edges
            uint2 ab = reinterpret_cast<const uint2 *>(rec + GSEG_REC_HEAD + 2 * (size_t)nV)[k];
            ab.x += jd.voff[s]; ab.y += jd.voff[s];
            B.eab[1][j] = ab;
            B.ew[1][j] = rec[GSEG_REC_HEAD + 2 * (size_t)nV + 2 * (size_t)nE + k];
            continue;
        }
        // cut edge between strip s (its bottom row) and strip s + 1 (its top row)
        const u32 *rec2 = recs + (size_t)(s + 1) * jd.stride_words;
        const u32 nV2 = jd.voff[s + 2] - jd.voff[s + 1], nE2 = jd.ne[s + 1];
        const u32 *bot_lab = rec + GSEG_REC_HEAD + 2 * (size_t)nV + 3 * (size_t)nE + w;
        const float *bot_col = reinterpret_cast<const float *>(bot_lab + w) + 3 * (size_t)w;
        const u32 *top_lab = rec2 + GSEG_REC_HEAD + 2 * (size_t)nV2 + 3 * (size_t)nE2;
        const float *top_col = reinterpret_cast<const float *>(top_lab + 2 * (size_t)w);
        const u32 c = k - nE;
        u32 a, b, xa, xb;
        bool a_is_bot = true;
        if (c < w) { xa = c; xb = c; }                              // S
        else if (c < 2 * w - 1) { xa = c - w; xb = xa + 1; }        // SE: (x, last row) -> (x + 1, first row)
        else { xa = c - (2 * w - 1); xb = xa + 1; a_is_bot = false; } // NE: (x, first row of s + 1) -> (x + 1, last row of s)
        float wv;
        if (a_is_bot) {
            a = bot_lab[xa] + jd.voff[s]; b = top_lab[xb] + jd.voff[s + 1];
            wv = l2_rn(bot_col[xa], bot_col[w + xa], bot_col[2 * (size_t)w + xa], top_col[xb], top_col[w + xb], top_col[2 * (size_t)w + xb]);
        } else {
            a = top_lab[xa] + jd.voff[s + 1]; b = bot_lab[xb] + jd.voff[s];
            wv = l2_rn(top_col[xa], top_col[w + xa], top_col[2 * (size_t)w + xa], bot_col[xb], bot_col[w + xb], bot_col[2 * (size_t)w + xb]);
        }
        B.eab[1][j] = make_uint2(a, b);
        B.ew[1][j] = __float_as_uint(wv);
    }
}
// final labels of a strip: joined-graph label of (strip-local dense id + the strip's id offset)
template <typename OutT>
__global__ void __launch_bounds__(NT) k_map_labels(const int *__restrict__ labels, const u32 *__restrict__ F, u32 off, size_t V,
                                                   OutT *__restrict__ out) {
    for (size_t p = (size_t)blockIdx.x * NT + threadIdx.x; p < V; p += (size_t)gridDim.x * NT) out[p] = (OutT)F[off + (u32)labels[p]];
}

// ------------------------------------------------------------------------------------------------
// a12: hierarchy materialisation.  Level l = composition of the maps of rounds 0..l.  OutT: int32, or
// uint16 / uint8 when the level has few enough components (the label image is most of what an end-to-end
// run sends back over PCIe).  Rounds whose map the host folded into an earlier one (map_skip) are passed over.
// ------------------------------------------------------------------------------------------------
template <typename OutT>
__global__ void __launch_bounds__(NT) k_compose(const GsegCtl *__restrict__ ctl, const u32 *__restrict__ arena,
                                                int last_round, OutT *__restrict__ out) {
    const u32 V0 = (u32)ctl->p.w * (u32)ctl->p.h;
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V0; p += gridDim.x * NT) {
        u32 l = arena[p];
        for (int r = 1; r <= last_round; ++r)
            if (!ctl->map_skip[r]) {
                GSEG_CHK(ctl, l < ctl->stV[r] && (unsigned long long)ctl->map_off[r] + l < ctl->p.arena_cap, 10);
                l = arena[ctl->map_off[r] + l];
            }
        out[p] = (OutT)l;
    }
}
// Arena compaction (FELZ): rounds 0..last folded into round 0's map in place.  A pixel's chase reads its own
// round-0 entry and entries of later maps only, so overwriting the round-0 entries as we go is safe.
__global__ void __launch_bounds__(NT) k_compose_inplace(const GsegCtl *ctl, u32 *arena, int last_round) {
    const u32 V0 = (u32)ctl->p.w * (u32)ctl->p.h;
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V0; p += gridDim.x * NT) {
        u32 l = arena[p];
        for (int r = 1; r <= last_round; ++r)
            if (!ctl->map_skip[r]) l = arena[ctl->map_off[r] + l];
        arena[p] = l;
    }
}
// Two-step form for deep hierarchies: the maps of rounds first..last act on few components, so they are
// composed once into a table F (n = components entering round `first`) ...
__global__ void __launch_bounds__(NT) k_compose_table(const GsegCtl *__restrict__ ctl, const u32 *__restrict__ arena,
                                                      int first, int last, u32 n, u32 *__restrict__ F) {
    for (u32 c = blockIdx.x * NT + threadIdx.x; c < n; c += gridDim.x * NT) {
        u32 l = c;
        for (int r = first; r <= last; ++r)
            if (!ctl->map_skip[r]) l = arena[ctl->map_off[r] + l];
        F[c] = l;
    }
}
// ... and every pixel chases only the early rounds 0..first-1 and then looks its label up in F.
template <typename OutT>
__global__ void __launch_bounds__(NT) k_compose_px(const GsegCtl *__restrict__ ctl, const u32 *__restrict__ arena,
                                                   int first, const u32 *__restrict__ F, OutT *__restrict__ out) {
    const u32 V0 = (u32)ctl->p.w * (u32)ctl->p.h;
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V0; p += gridDim.x * NT) {
        u32 l = arena[p];
        for (int r = 1; r < first; ++r)
            if (!ctl->map_skip[r]) l = arena[ctl->map_off[r] + l];
        out[p] = (OutT)F[l];
    }
}
// one more level from the previous one (all-levels output: V reads + V writes per level)
__global__ void __launch_bounds__(NT) k_compose_step(const GsegCtl *__restrict__ ctl, const u32 *__restrict__ arena,
                                                     int round, const int *__restrict__ prev, int *__restrict__ out) {
    const u32 V0 = (u32)ctl->p.w * (u32)ctl->p.h;
    const u32 *map = arena + ctl->map_off[round];
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V0; p += gridDim.x * NT) out[p] = (int)map[prev[p]];
}

__device__ __forceinline__ u64 d_sm64(u64 x) {
    u64 z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ u64 d_hash2(u64 seed, u64 a, u64 b) {
    return d_sm64(d_sm64(seed ^ (a * 0xD6E8FEB86659FD93ull)) + b);
}

// a14: random colour per component id (counter-based hash instead of cuRAND state).
__global__ void __launch_bounds__(NT) k_colorize(const int *__restrict__ labels, u32 V0, u64 seed,
                                                 uint8_t *__restrict__ out) {
    for (u32 p = blockIdx.x * NT + threadIdx.x; p < V0; p += gridDim.x * NT) {
        const u64 hsh = d_hash2(seed, (u64)(u32)labels[p], 3);
        out[3 * (size_t)p] = (uint8_t)(hsh & 255);
        out[3 * (size_t)p + 1] = (uint8_t)((hsh >> 8) & 255);
        out[3 * (size_t)p + 2] = (uint8_t)((hsh >> 16) & 255);
    }
}

// Synthetic input generator (SURVEY.md section 8d); integer arithmetic only.
// Rows [y_first, y_first + h) of the image of width w (a pixel depends on its coordinates and the seed only, so a
// strip of a larger image can be generated on its own).
__global__ void __launch_bounds__(NT) k_synth(uint8_t *__restrict__ rgb, int w, int h, u64 seed, int y_first) {
    const size_t V = (size_t)w * (size_t)h;
    for (size_t p = (size_t)blockIdx.x * NT + threadIdx.x; p < V; p += (size_t)gridDim.x * NT) {
        const int y = (int)(p / (size_t)w) + y_first, x = (int)(p % (size_t)w);
        const int cx = x >> 6, cy = y >> 6;
        long long bestd = 0x7FFFFFFFFFFFFFFFll;
        u64 besth = 0;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const int ccx = cx + dx, ccy = cy + dy;
                const u64 cell = ((u64)(ccy + 1) << 20) | (u64)(ccx + 1);
                const u64 hs = d_hash2(seed, cell, 1);
                const long long sx = (long long)ccx * 64 + (long long)(hs & 63);
                const long long sy = (long long)ccy * 64 + (long long)((hs >> 6) & 63);
                const long long d = (x - sx) * (x - sx) + (y - sy) * (y - sy);
                if (d < bestd) { bestd = d; besth = hs; }
            }
        const u64 hn = d_hash2(seed, (u64)y * (u64)w + (u64)x, 2);
        for (int c = 0; c < 3; ++c) {
            const int base = (int)((besth >> (16 + 8 * c)) & 255);
            const int n = (int)(((hn >> (16 * c)) & 0xFFFF) % 17) - 8;
            rgb[3 * p + c] = (uint8_t)min(max(base + n, 0), 255);
        }
    }
}
