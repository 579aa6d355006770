// tsd_kernels.cuh -- hand-written sm_100a kernels of the candidate-window scoring and recognition path.
//
// One kernel per stage (BASELINE.json north_star).  Citations: DET = "Deteción de Objetos/source.py",
// REC = "Reconocimiento de Objetos/source.py" of the reference; the cv2 / sklearn internals each kernel reproduces
// are specified in SURVEY.md Appendix A.  Compiled with -fmad=false: f64/f32 steps round like the reference's
// scalar numpy / OpenCV code (no FMA contraction).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <float.h>

#ifndef TSD_K2_UNROLL
#define TSD_K2_UNROLL 3          // destination rows of the K2 general path per trip (all their loads in flight together; measured at 4096 frames, wide loads: 2: .780, 3: .758, 4: .821, 5: .98 ms with 40 registers)
#endif
#ifndef TSD_K3_UNROLL
#define TSD_K3_UNROLL 4          // pixels per lane in flight in the mask kernel
#endif
#ifndef TSD_HIST_GRID
#define TSD_HIST_GRID 64         // persistent CTAs per SM of k5_hist
#endif
#ifndef TSD_K3_GRID
#define TSD_K3_GRID 32           // persistent CTAs per SM of k3_masks
#endif
#ifndef TSD_FOLD_WARPS
#define TSD_FOLD_WARPS 4         // warps (= frames in flight) per CTA of the warp-per-frame fold
#endif
#ifndef TSD_FOLD_MINB
#define TSD_FOLD_MINB 1          // min resident CTAs per SM of the warp-per-frame fold (register budget: 1 -> as many as it likes, 128)
#endif
#ifndef TSD_HIST_UNROLL
#define TSD_HIST_UNROLL 8        // pixels per lane in flight in the two histogram passes (measured: 2: .266, 4: .274, 5: .283, 7-8: .259, 10: .310, 20: .369 ms)
#endif

#ifndef TSD_HIST_MINB
#define TSD_HIST_MINB 8          // min resident CTAs per SM of k5_hist (register budget: 8 -> 64 registers)
#endif
#ifndef TSD_K2_MINB
#define TSD_K2_MINB 12           // min resident CTAs per SM of k2_crop_resize_v2 (12 -> 40 registers)
#endif
#ifndef TSD_K2_WIDE
#define TSD_K2_WIDE 1            // K2 general path: aligned 32-bit tap loads + IDP.2A horizontal pass (0: byte loads)
#endif
#ifndef TSD_HIST_GROUP_UNROLL
#define TSD_HIST_GROUP_UNROLL 2  // groups of 4 pixels per lane in flight in the aligned histogram passes (measured at 4096 frames: 1: .922, 2: .921, 3: .934, 4: .953 ms)
#endif

namespace tsd {
constexpr int kHistGroupUnroll = TSD_HIST_GROUP_UNROLL;
constexpr int kK2Unroll = TSD_K2_UNROLL, kHistUnroll = TSD_HIST_UNROLL, kK3Unroll = TSD_K3_UNROLL;     // (#pragma unroll takes a constant expression, not a macro)

constexpr int kHistH = 50, kHistS = 60, kHistBins = kHistH * kHistS;   // DET:578
constexpr int kMaxD = 32;
constexpr int kMaxPx = kMaxD * kMaxD;

// Internal layouts are padded so that every window / sparse histogram starts on a 16-byte boundary (128-bit loads):
// window stride = D*D*C bytes rounded up to 16 (1875 -> 1888; pad bytes are ZERO), entry stride = D*D words rounded up to 4.
__host__ __device__ inline int win_stride(int npx, int C) { return (npx * C + 15) & ~15; }
__host__ __device__ inline int ent_stride(int npx) { return (npx + 3) & ~3; }

// order-independent pixel-content hash: sum over pixels of mix(position, bgr).  Equal windows -> equal hash; used only as a
// pre-filter of the pop-by-pixel-equality rule (DET:471-477), candidates are always verified byte by byte.
__device__ __forceinline__ uint32_t pix_hash32(int p, uint32_t bgr) {
    const uint32_t x = bgr * 0x9E3779B1u + (uint32_t)p * 0x85EBCA6Bu;       // two IMADs; p * K strength-reduces to an add in the pixel loops
    return x ^ (x >> 15);
}

// ---- small tables (global memory, L2-resident; staged to shared memory by the kernels that index them per lane)
struct Tables {
    int32_t sdiv[256];      // rne((255<<12)/i)         OpenCV RGB2HSV_b
    int32_t hdiv[256];      // rne((180<<12)/(6 i))
    uint8_t hbin[256];      // floor(H * 50/180)        calcHist LUT (only 0..179 used)
    uint8_t sbin[256];      // floor(S * 60/256)
};

struct HsvBounds {          // DET:70-86
    uint8_t red_lo[2][3], red_hi[2][3], blue_lo[3], blue_hi[3];
};

__device__ __forceinline__ void bgr2hsv(int b, int g, int r, const int32_t* __restrict__ sdiv,
                                        const int32_t* __restrict__ hdiv, int& H, int& S, int& V) {
    int v = max(b, max(g, r)), m = min(b, min(g, r));
    int d = v - m;
    int h = (v == r) ? (g - b) : (v == g) ? (b - r + 2 * d) : (r - g + 4 * d);
    S = (d * sdiv[v] + (1 << 11)) >> 12;
    h = (h * hdiv[d] + (1 << 11)) >> 12;
    H = h < 0 ? h + 180 : h;
    V = v;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- exclusive scan of per-frame counts by the LAST CTA of a grid to finish -----------------------------------------------------
// The per-frame counts of a stage (aspect-passing windows, survivors, detections) are turned into CSR offsets by whichever CTA of
// the producing kernel retires last, instead of by a separate single-CTA launch: the chains of small batches (real MSER frames:
// ~35 boxes per frame) are bound by launch latency, not by work.  `ticket` is a zero-initialised counter that is reset on the way out.
__device__ __forceinline__ void block_scan_offsets(const int32_t* counts, int n, int32_t* offsets) {
    __shared__ int32_t s_wsum[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = (blockDim.x + 31) >> 5;
    const int per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
    const int b = min(n, tid * per), e = min(n, b + per);
    int sum = 0;
    for (int i = b; i < e; i++) sum += __ldcg(counts + i);   // (written by other SMs in this launch: not through L1)
    int x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) s_wsum[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int v = lane < nw ? s_wsum[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += y; }
        s_wsum[lane] = v;
    }
    __syncthreads();
    int run = (wid ? s_wsum[wid - 1] : 0) + x - sum;
    for (int i = b; i < e; i++) { offsets[i] = run; run += __ldcg(counts + i); }
    if (tid == (int)blockDim.x - 1) offsets[n] = s_wsum[nw - 1];
}

// Call at the very end of a kernel, by all threads of every CTA (after the CTA's counts are written).
__device__ __forceinline__ void scan_by_last_block(const int32_t* counts, int n, int32_t* offsets, unsigned* ticket) {
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    block_scan_offsets(counts, n, offsets);
    if (threadIdx.x == 0) *ticket = 0;
}

// =====================================================================================================
// K1  makeWindowBiggerOrDiscardFakeDetections  (DET:155-174 = REC:88-107), SURVEY A.1.  f64, no FMA.
// =====================================================================================================
__device__ __forceinline__ bool expand_box(int4 b, double pm1, double alo, double ahi, int4& out) {
    double w = (double)b.z, h = (double)b.w;
    double ratio = __ddiv_rn(w, h);
    if (!(alo < ratio && ratio < ahi)) return false;
    double dw = __dmul_rn(__dmul_rn(w, pm1), 0.5), dh = __dmul_rn(__dmul_rn(h, pm1), 0.5);
    double x1 = __dsub_rn((double)b.x, dw), y1 = __dsub_rn((double)b.y, dh);
    double x2 = __dadd_rn((double)(b.x + b.z), dw), y2 = __dadd_rn((double)(b.y + b.w), dh);
    x1 = x1 > 0 ? x1 : 0; y1 = y1 > 0 ? y1 : 0; x2 = x2 > 0 ? x2 : 0; y2 = y2 > 0 ? y2 : 0;
    out = make_int4((int)x1, (int)y1, (int)x2, (int)y2);     // int(): truncation
    return true;
}

// one result per box (per-stage parity entry point tsd_expand_boxes)
__global__ void k1_expand_kernel(const int4* __restrict__ boxes, int n, double pm1, double alo, double ahi,
                                 int4* __restrict__ coords, uint8_t* __restrict__ valid) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int4 c = make_int4(0, 0, 0, 0);
    bool ok = expand_box(boxes[i], pm1, alo, ahi, c);
    coords[i] = c;
    valid[i] = ok ? 1 : 0;
}

// per frame: count of aspect-passing boxes whose (frame-clipped) crop is not empty.  One warp per frame.
// The last CTA to finish turns the counts into the CSR offsets of the windows (win_offsets [nframes + 1]).
__global__ void k1_count_kernel(const int4* __restrict__ boxes, const int32_t* __restrict__ box_offsets, int nframes,
                                int H, int W, double pm1, double alo, double ahi, int32_t* __restrict__ counts,
                                int32_t* __restrict__ win_offsets, unsigned* __restrict__ ticket) {
    int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f < nframes) {
        int b0 = box_offsets[f], b1 = box_offsets[f + 1], cnt = 0;
        for (int i = b0 + lane; i < b1; i += 32) {
            int4 c;
            if (expand_box(boxes[i], pm1, alo, ahi, c) && min(c.z, W) > min(c.x, W) && min(c.w, H) > min(c.y, H)) cnt++;
        }
        cnt = warp_sum_i(cnt);
        if (lane == 0) counts[f] = cnt;
    }
    scan_by_last_block(counts, nframes, win_offsets, ticket);
}

// order-preserving compaction: coords of passing boxes -> coords[win_offsets[f] + rank], win_frame[...] = f.
__global__ void k1_compact_kernel(const int4* __restrict__ boxes, const int32_t* __restrict__ box_offsets, int nframes,
                                  int H, int W, double pm1, double alo, double ahi,
                                  const int32_t* __restrict__ win_offsets, int4* __restrict__ coords,
                                  int32_t* __restrict__ win_frame) {
    int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f >= nframes) return;
    int b0 = box_offsets[f], b1 = box_offsets[f + 1], out = win_offsets[f];
    for (int base = b0; base < b1; base += 32) {
        int i = base + lane;
        int4 c = make_int4(0, 0, 0, 0);
        bool ok = false;
        if (i < b1) ok = expand_box(boxes[i], pm1, alo, ahi, c) && min(c.z, W) > min(c.x, W) && min(c.w, H) > min(c.y, H);
        unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            int r = out + __popc(m & ((1u << lane) - 1));
            coords[r] = c;
            win_frame[r] = f;
        }
        out += __popc(m);
    }
}

// =====================================================================================================
// K2  cv2.resize(cropImageByCoords(coords, frame), (D, D))  (DET:123-124,570-572; REC:57,253-254), SURVEY A.2.
// One warp per window.  The crop is the numpy slice frame[y1:y2, x1:x2] clipped to the frame; three code paths:
// same-size copy, exact 2x2 INTER_AREA, general two-pass 11-bit fixed point (x coefficient clamp, y row clip).
// v1: taps are gathered straight from global memory through L1 (a window's ROI is ~5 KB and stays L1-resident).
// =====================================================================================================
template <int C>
__global__ void __launch_bounds__(128) k2_crop_resize_kernel(
    const uint8_t* __restrict__ frames, int H, int W, int64_t row_stride, int64_t frame_stride,
    const int4* __restrict__ coords, const int32_t* __restrict__ win_frame, const int32_t* __restrict__ n_ptr, int n_max,
    int D, uint8_t* __restrict__ windows, int out_stride) {
    __shared__ int16_t s_xo[4][kMaxD], s_xa0[4][kMaxD], s_xa1[4][kMaxD];
    __shared__ int16_t s_y0[4][kMaxD], s_y1[4][kMaxD], s_yb0[4][kMaxD], s_yb1[4][kMaxD];
    const int wl = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = blockIdx.x * 4 + wl;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    if (w >= n) return;
    const int4 c = coords[w];
    const int cx = min(c.x, W), cy = min(c.y, H);
    const int cw = min(c.z, W) - cx, ch = min(c.w, H) - cy;
    const uint8_t* __restrict__ src = frames + (int64_t)win_frame[w] * frame_stride + (int64_t)cy * row_stride + (int64_t)cx * C;
    uint8_t* __restrict__ dst = windows + (int64_t)w * out_stride;
    const int rowlen = D * C, total = D * rowlen;
    if (cw <= 0 || ch <= 0) {                                // empty crop (cv2.resize would raise; K1 never emits one): a defined, all-zero window
        for (int i = lane; i < out_stride; i += 32) dst[i] = 0;
        return;
    }
    for (int i = total + lane; i < out_stride; i += 32) dst[i] = 0;     // pad bytes of the internal layout are zero
    if (cw == D && ch == D) {                               // same size: copy
        for (int i = lane; i < total; i += 32) { int y = i / rowlen, r = i - y * rowlen; dst[i] = src[(int64_t)y * row_stride + r]; }
        return;
    }
    if (cw == 2 * D && ch == 2 * D) {                       // INTER_AREA 2x2 fast path
        for (int i = lane; i < total; i += 32) {
            int y = i / rowlen, r = i - y * rowlen, x = r / C, k = r - x * C;
            const uint8_t* p = src + (int64_t)(2 * y) * row_stride + (2 * x) * C + k;
            dst[i] = (uint8_t)((p[0] + p[C] + p[row_stride] + p[row_stride + C] + 2) >> 2);
        }
        return;
    }
    if (lane < D) {                                         // coefficient tables (float32 rounding as in OpenCV)
        {
            double scale = 1.0 / ((double)D / (double)cw);
            float f = (float)(((double)lane + 0.5) * scale - 0.5);
            int s = (int)floorf(f); f -= (float)s;
            if (s < 0) { f = 0.f; s = 0; }
            if (s >= cw - 1) { f = 0.f; s = cw - 1; }
            s_xo[wl][lane] = (int16_t)s;
            s_xa0[wl][lane] = (int16_t)__float2int_rn((1.f - f) * 2048.f);
            s_xa1[wl][lane] = (int16_t)__float2int_rn(f * 2048.f);
        }
        {
            double scale = 1.0 / ((double)D / (double)ch);
            float f = (float)(((double)lane + 0.5) * scale - 0.5);
            int s = (int)floorf(f); f -= (float)s;
            s_y0[wl][lane] = (int16_t)min(max(s, 0), ch - 1);
            s_y1[wl][lane] = (int16_t)min(max(s + 1, 0), ch - 1);
            s_yb0[wl][lane] = (int16_t)__float2int_rn((1.f - f) * 2048.f);
            s_yb1[wl][lane] = (int16_t)__float2int_rn(f * 2048.f);
        }
    }
    __syncwarp();
    for (int i = lane; i < total; i += 32) {
        int y = i / rowlen, r = i - y * rowlen, x = r / C, k = r - x * C;
        int s0 = s_xo[wl][x], s1 = min(s0 + 1, cw - 1);
        int a0 = s_xa0[wl][x], a1 = s_xa1[wl][x];
        const uint8_t* S0 = src + (int64_t)s_y0[wl][y] * row_stride;
        const uint8_t* S1 = src + (int64_t)s_y1[wl][y] * row_stride;
        int t0 = S0[s0 * C + k] * a0 + S0[s1 * C + k] * a1;
        int t1 = S1[s0 * C + k] * a0 + S1[s1 * C + k] * a1;
        int v = (((s_yb0[wl][y] * (t0 >> 4)) >> 16) + ((s_yb1[wl][y] * (t1 >> 4)) >> 16) + 2) >> 2;
        dst[i] = (uint8_t)v;
    }
}

// K2 v2: same arithmetic, restructured for instruction count (v1 was issue-bound at ~100 instructions per output
// byte-iteration).  One warp per window, lane = destination column; the x coefficients live in registers, the y
// coefficients are computed by lane dy and broadcast through shared memory; each lane walks the D destination rows and reads its
// 2 x 2 taps x C channels straight from the frame through L1 (one row segment per load): as aligned 32-bit words + IDP.2A for
// BGR frames with 4-byte aligned rows (k2_rows_wide), as byte loads otherwise (k2_rows).  Persistent warps stride over the windows.
// (Variants that lost on B200 -- crop staged in shared memory with cp.async or by TMA, row reuse + staged output, one CTA per
// frame, L2 prefetch of the ROI -- are documented with their measurements in DESIGN.md section 8.)
// Which windows the TMA-staged resize kernel takes (tsd_k2_tma.cuh): crops whose byte span, widened to whole 16-byte units in front
// and 64-byte units in total, and whose rows, in boxes of 8, fit the per-warp staging buffer.  cx = clipped x1, cw / ch = clipped size.
constexpr int kTmaStageBytes = 10240;
constexpr int kTmaBoxRows = 8;
__device__ __forceinline__ bool k2_tma_takes(int cx, int cw, int ch) {
    const int P = ((cw * 3 + ((cx * 3) & 15) + 63) >> 6) << 6, nops = (ch + kTmaBoxRows - 1) / kTmaBoxRows;
    return cw > 0 && ch > 0 && P <= 256 && ch <= 64 && P * kTmaBoxRows * nops <= kTmaStageBytes;
}

// The D destination rows of one window in the general (two-pass 11-bit fixed point) case.  XDC: the second tap sits C bytes after the
// first in every column (xd1 == C, true for every crop wider than D).  (v0 >> 16) + (v1 >> 16) + 2 is folded into one multiply-add:
// ((v1 + (2 << 16)) >> 16) == (v1 >> 16) + 2.
template <int C, int D, bool XDC>
__device__ __forceinline__ void k2_rows(const uint8_t* __restrict__ px, const int4* s_y, int xd1, int xa0, int xa1, uint8_t* __restrict__ dst, bool act) {
#pragma unroll kK2Unroll
    for (int dy = 0; dy < D; dy++) {
        const int4 yc = s_y[dy];
        const int b0 = yc.z, b1 = yc.w;
        const uint8_t* p0 = px + (uint32_t)yc.x;
        const uint8_t* p1 = px + (uint32_t)yc.y;
        const uint8_t* q0 = XDC ? p0 + C : p0 + xd1;
        const uint8_t* q1 = XDC ? p1 + C : p1 + xd1;
        int v[C];
#pragma unroll
        for (int k = 0; k < C; k++) {
            const int t0 = __ldg(p0 + k) * xa0 + __ldg(q0 + k) * xa1;
            const int t1 = __ldg(p1 + k) * xa0 + __ldg(q1 + k) * xa1;
            v[k] = (((b0 * (t0 >> 4)) >> 16) + ((b1 * (t1 >> 4) + (2 << 16)) >> 16)) >> 2;
        }
        if (act) {
#pragma unroll
            for (int k = 0; k < C; k++) dst[dy * D * C + k] = (uint8_t)v[k];
        }
    }
}

// The same rows with WIDE loads (C = 3, 4-byte aligned frames and strides): the 6 consecutive bytes a lane needs of a source row (two
// taps x three channels) come from 2-3 aligned 32-bit loads instead of 6 byte loads (the byte-load kernel keeps the L1 data pipe
// ~70 % busy: 645 wavefronts per window), a funnel shift brings them to bit 0, two byte permutes pair each channel's taps and one
// IDP.2A per channel (16-bit coefficients x 8-bit taps) is the horizontal pass.  The second tap is read at +3 bytes in every
// column: where cv2 clamps it onto the first (x = 0 of an up-scale, the last column) its coefficient is 0.  An aligned word may reach
// up to 6 bytes past the bytes needed, so a window on the last row of the last frame takes the byte loads.
template <int D>
__device__ __forceinline__ void k2_rows_wide(const uint8_t* __restrict__ px, const int4* s_y, int xa0, int xa1, uint8_t* dst, bool act) {
    const unsigned o = (unsigned)(reinterpret_cast<uintptr_t>(px) & 3);
    const unsigned o8 = o * 8;
    const uint8_t* pa = px - o;
    asm volatile("" : "+l"(pa), "+l"(dst));                  // both stay in registers: one 64-bit add per row pointer, immediate store offsets
    const bool third = o == 3;                               // bytes o .. o+5 of the aligned words: a third word only from offset 3
    const unsigned xa = (unsigned)xa0 | ((unsigned)xa1 << 16);
    // kK2Unroll destination rows per trip: all their loads are issued before the first result is stored
    for (int dy0 = 0; dy0 < D; dy0 += kK2Unroll) {
        uint32_t a0[kK2Unroll], a1[kK2Unroll], a2[kK2Unroll], c0[kK2Unroll], c1[kK2Unroll], c2[kK2Unroll];
        int b0[kK2Unroll], b1[kK2Unroll];
#pragma unroll
        for (int u = 0; u < kK2Unroll; u++) {
            const int4 yc = s_y[min(dy0 + u, D - 1)];
            b0[u] = yc.z; b1[u] = yc.w;
            const uint32_t* q0 = reinterpret_cast<const uint32_t*>(pa + (uint32_t)yc.x);
            const uint32_t* q1 = reinterpret_cast<const uint32_t*>(pa + (uint32_t)yc.y);
            a0[u] = __ldg(q0); a1[u] = __ldg(q0 + 1); a2[u] = third ? __ldg(q0 + 2) : 0u;
            c0[u] = __ldg(q1); c1[u] = __ldg(q1 + 1); c2[u] = third ? __ldg(q1 + 2) : 0u;
        }
#pragma unroll
        for (int u = 0; u < kK2Unroll; u++) {
            const int dy = dy0 + u;
            const uint32_t lo0 = __funnelshift_r(a0[u], a1[u], o8), hi0 = __funnelshift_r(a1[u], a2[u], o8);      // bytes 0-3 / 4-7 counted from the first tap
            const uint32_t lo1 = __funnelshift_r(c0[u], c1[u], o8), hi1 = __funnelshift_r(c1[u], c2[u], o8);
            const uint32_t bg0 = __byte_perm(lo0, hi0, 0x4130), r0 = __byte_perm(lo0, hi0, 0x0052);               // [B0 B1 G0 G1], [R0 R1 . .]
            const uint32_t bg1 = __byte_perm(lo1, hi1, 0x4130), r1 = __byte_perm(lo1, hi1, 0x0052);
            int v[3];
            {
                const int t0 = (int)__dp2a_lo(xa, bg0, 0u), t1 = (int)__dp2a_lo(xa, bg1, 0u);
                v[0] = (((b0[u] * (t0 >> 4)) >> 16) + ((b1[u] * (t1 >> 4) + (2 << 16)) >> 16)) >> 2;
            }
            {
                const int t0 = (int)__dp2a_hi(xa, bg0, 0u), t1 = (int)__dp2a_hi(xa, bg1, 0u);
                v[1] = (((b0[u] * (t0 >> 4)) >> 16) + ((b1[u] * (t1 >> 4) + (2 << 16)) >> 16)) >> 2;
            }
            {
                const int t0 = (int)__dp2a_lo(xa, r0, 0u), t1 = (int)__dp2a_lo(xa, r1, 0u);
                v[2] = (((b0[u] * (t0 >> 4)) >> 16) + ((b1[u] * (t1 >> 4) + (2 << 16)) >> 16)) >> 2;
            }
            if (act && dy < D) {
#pragma unroll
                for (int k = 0; k < 3; k++) dst[dy * D * 3 + k] = (uint8_t)v[k];
            }
        }
    }
}

// One window by one warp, taps gathered straight from the frame (the body of k2_crop_resize_v2; also the path k2_crop_resize_tma
// takes for crops that do not fit its staging buffer).  s_y = the warp's 32 x int4 scratch.
template <int C, int D>
__device__ __forceinline__ void k2_window_gather(const uint8_t* __restrict__ frames, int H, int W, int64_t row_stride, int64_t frame_stride,
                                                 const int4* __restrict__ coords, const int32_t* __restrict__ win_frame, int w,
                                                 uint8_t* __restrict__ windows, int out_stride, int4* s_y, int wide_last = -2) {
    const int lane = threadIdx.x & 31;
    const int4 c = coords[w];
    const int cx = min(c.x, W), cy = min(c.y, H);
    const int cw = min(c.z, W) - cx, ch = min(c.w, H) - cy;
    if (cw <= 0 || ch <= 0) {                                // empty crop (cv2.resize would raise; K1 never emits one): a defined, all-zero window
        for (int i = lane; i < out_stride; i += 32) windows[(int64_t)w * out_stride + i] = 0;
        return;
    }
    const uint8_t* __restrict__ src = frames + (int64_t)win_frame[w] * frame_stride + (int64_t)cy * row_stride + (int64_t)cx * C;
    uint8_t* __restrict__ dst = windows + (int64_t)w * out_stride + lane * C;
    if (D * D * C + lane < out_stride) windows[(int64_t)w * out_stride + D * D * C + lane] = 0;    // zero pad (< 16 bytes)
    const bool act = lane < D;
    const int li = act ? lane : 0;
    if (cw == D && ch == D) {                               // same size: copy
        const uint8_t* p = src + li * C;
#pragma unroll 5
        for (int dy = 0; dy < D; dy++) {
            uint8_t v[C];
#pragma unroll
            for (int k = 0; k < C; k++) v[k] = __ldg(p + (int64_t)dy * row_stride + k);
            if (act) {
#pragma unroll
                for (int k = 0; k < C; k++) dst[dy * D * C + k] = v[k];
            }
        }
        return;
    }
    if (cw == 2 * D && ch == 2 * D) {                       // INTER_AREA 2x2 fast path
        const uint8_t* p = src + 2 * li * C;
#pragma unroll 5
        for (int dy = 0; dy < D; dy++) {
            const uint8_t* q0 = p + (int64_t)(2 * dy) * row_stride;
            const uint8_t* q1 = q0 + row_stride;
            int v[C];
#pragma unroll
            for (int k = 0; k < C; k++) v[k] = (__ldg(q0 + k) + __ldg(q0 + C + k) + __ldg(q1 + k) + __ldg(q1 + C + k) + 2) >> 2;
            if (act) {
#pragma unroll
                for (int k = 0; k < C; k++) dst[dy * D * C + k] = (uint8_t)v[k];
            }
        }
        return;
    }
    // coefficient tables (float32 rounding as in OpenCV); lane doubles as dx (x tables) and as dy (y tables)
    int xs0, xd1, xa0, xa1, yr0, yr1, yb0, yb1;
    {
        const double scale = 1.0 / ((double)D / (double)cw);
        float f = (float)(((double)li + 0.5) * scale - 0.5);
        int s = (int)floorf(f); f -= (float)s;
        if (s < 0) { f = 0.f; s = 0; }
        if (s >= cw - 1) { f = 0.f; s = cw - 1; }
        xs0 = s * C;
        xd1 = (min(s + 1, cw - 1) - s) * C;
        xa0 = __float2int_rn((1.f - f) * 2048.f);
        xa1 = __float2int_rn(f * 2048.f);
    }
    {
        const double scale = 1.0 / ((double)D / (double)ch);
        float f = (float)(((double)li + 0.5) * scale - 0.5);
        int s = (int)floorf(f); f -= (float)s;
        yr0 = min(max(s, 0), ch - 1);
        yr1 = min(max(s + 1, 0), ch - 1);
        yb0 = __float2int_rn((1.f - f) * 2048.f);
        yb1 = __float2int_rn(f * 2048.f);
    }
    const uint8_t* px = src + xs0;
    __syncwarp();                                            // (the previous window's rows are consumed)
    // one 128-bit broadcast read per destination row instead of 4 shuffles; the rows travel as 32-bit BYTE offsets (the host checks
    // that a frame spans less than 2 GiB), so a tap address is one 64-bit add instead of a 64-bit multiply-add per row
    s_y[lane] = make_int4(yr0 * (int)row_stride, yr1 * (int)row_stride, yb0, yb1);
    __syncwarp();
    // every down-scale (cw > D) has its second tap exactly one pixel to the right in every column: the tap offsets are immediates
    if (C == 3 && TSD_K2_WIDE && wide_last >= -1 && !(win_frame[w] == wide_last && cy + ch == H)) k2_rows_wide<D>(px, s_y, xa0, xa1, dst, act);
    else if (__all_sync(0xffffffffu, xd1 == C)) k2_rows<C, D, true>(px, s_y, C, xa0, xa1, dst, act);
    else k2_rows<C, D, false>(px, s_y, xd1, xa0, xa1, dst, act);
}

template <int C, int D>
__global__ void __launch_bounds__(128, TSD_K2_MINB) k2_crop_resize_v2_kernel(
    const uint8_t* __restrict__ frames, int H, int W, int64_t row_stride, int64_t frame_stride,
    const int4* __restrict__ coords, const int32_t* __restrict__ win_frame, const int32_t* __restrict__ n_ptr, int n_max,
    uint8_t* __restrict__ windows, int out_stride, int skip_tma, int wide_last) {
    __shared__ int4 s_y[4][32];                              // per warp: (row0, row1, weight0, weight1) of every destination row
    const int wl = threadIdx.x >> 5;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += nwarps) {     // (the grid normally covers all windows: one trip)
        if (skip_tma) {                                      // the TMA-staged kernel, launched beside this one, takes the crops that fit its buffer
            const int4 c = coords[w];
            const int cx = min(c.x, W), cy = min(c.y, H);
            if (k2_tma_takes(cx, min(c.z, W) - cx, min(c.w, H) - cy)) continue;
        }
        k2_window_gather<C, D>(frames, H, W, row_stride, frame_stride, coords, win_frame, w, windows, out_stride, s_y[wl], wide_last);
    }
}

// =====================================================================================================
// Host-frame staging (tsd_detect_frames on PAGE-LOCKED host frames).  The candidate ROIs cover ~10 % of a frame, so copying whole
// frames wastes PCIe; letting K2 gather straight from host memory (round 1) fetched every 32-byte sector once per window that
// touches it (nested / jittered MSER boxes overlap heavily) and in requests as the taps happen to fall.  Instead:
//   stage_mark : one warp per window sets, in a per-frame bitmap over (row, 32-byte sector), every sector K2 will read -- the whole
//                byte span [3 x1, 3 x2) of each source row the resize touches (all rows of the crop up to 2D rows, else the two rows
//                per destination row, computed exactly like K2 does);
//   stage_copy : walks the bitmaps; lane l of a warp copies sector 32 w + l of bitmap word w when its bit is set, so runs of set bits
//                become coalesced 128-byte reads over PCIe, and every sector crosses the bus ONCE per batch; the copy lands in a
//                device-resident mirror with the frame's own layout, which K2 then reads at HBM speed.
// The mirror is never cleared: K2 only reads sectors that were marked (and therefore copied) in the same batch.
// =====================================================================================================
// gran = sectors per PCIe request unit (1, 2 or 4): the span is widened to whole units of 32 * gran bytes (a read request that
// fills a whole 128-byte line moves more payload per PCIe packet than four 32-byte ones).
__global__ void __launch_bounds__(128) stage_mark_kernel(const int4* __restrict__ coords, const int32_t* __restrict__ win_frame,
                                                         const int32_t* __restrict__ n_ptr, int n_max, int H, int W, int D, int wpr, int gran,
                                                         uint32_t* __restrict__ bitmap) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    if (w >= n) return;
    const int4 c = coords[w];
    const int cx = min(c.x, W), cy = min(c.y, H);
    const int cw = min(c.z, W) - cx, ch = min(c.w, H) - cy;
    if (cw <= 0 || ch <= 0) return;
    const int s0 = ((3 * cx) >> 5) & ~(gran - 1), s1 = min(((3 * (cx + cw) - 1) >> 5) | (gran - 1), ((3 * W + 31) >> 5) - 1);   // first / last 32-byte sector of the row span
    uint32_t* fb = bitmap + (int64_t)win_frame[w] * H * wpr;
    int rows[2], nrows = 0;
    if (ch <= 2 * D) {                                       // every row of the crop (copy / 2x2 AREA / down-scales up to 2)
        if (lane < ch) rows[nrows++] = cy + lane;
        if (lane + 32 < ch) rows[nrows++] = cy + lane + 32;
    } else if (lane < D) {                                   // the two source rows of destination row `lane` (same float steps as K2)
        const double scale = 1.0 / ((double)D / (double)ch);
        float f = (float)(((double)lane + 0.5) * scale - 0.5);
        const int sy = (int)floorf(f);
        rows[nrows++] = cy + min(max(sy, 0), ch - 1);
        rows[nrows++] = cy + min(max(sy + 1, 0), ch - 1);
    }
    for (int k = 0; k < nrows; k++) {
        uint32_t* rb = fb + (int64_t)rows[k] * wpr;
        for (int wd = s0 >> 5; wd <= (s1 >> 5); wd++) {
            const int lo = max(s0, 32 * wd) & 31, hi = min(s1, 32 * wd + 31) & 31;
            const uint32_t m = (hi == 31 ? 0xffffffffu : ((2u << hi) - 1u)) & ~((1u << lo) - 1u);
            if ((rb[wd] & m) != m) atomicOr(rb + wd, m);     // (most windows re-mark sectors an overlapping window already set)
        }
    }
}

// total words = nframes * H * wpr.  src rows: row_bytes valid bytes (a multiple of 16), 16-byte aligned base and strides (host checks).
// Four non-empty bitmap words per trip: all their loads are issued before the first store, so a warp keeps up to 8 x 16 bytes per
// lane in flight over PCIe (the copy is bound by the number of outstanding read requests, not by their size: a 128-byte L2 fetch
// hint and spans widened to whole 128-byte lines both measured slower, DESIGN.md section 8).
__global__ void __launch_bounds__(256) stage_copy_kernel(const uint8_t* __restrict__ src, int64_t row_stride, int64_t frame_stride, int H, int row_bytes,
                                                         int wpr, int64_t nwords, const uint32_t* __restrict__ bitmap, uint8_t* __restrict__ mirror,
                                                         unsigned long long* __restrict__ bytes_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long copied = 0;
    for (int64_t base = warp * 32; base < nwords; base += nwarps * 32) {
        const int64_t wi = base + lane;
        const uint32_t mine = wi < nwords ? __ldg(bitmap + wi) : 0u;
        unsigned nz = __ballot_sync(0xffffffffu, mine != 0u);
        while (nz) {
            int64_t o[4];
            int nb[4];                                       // bytes this lane copies for word u: 0, 16 or 32
#pragma unroll
            for (int u = 0; u < 4; u++) {
                nb[u] = 0; o[u] = 0;
                if (nz) {                                    // (warp-uniform)
                    const int k = __ffs(nz) - 1;
                    nz &= nz - 1;
                    const uint32_t wv = __shfl_sync(0xffffffffu, mine, k);
                    const int64_t g = base + k;              // global word index -> (frame, row, word of the row)
                    const int64_t fr = g / wpr;
                    const int wd = (int)(g - fr * wpr);
                    const int64_t f = fr / H;
                    const int row = (int)(fr - f * H);
                    const int off = (32 * wd + lane) * 32;   // byte offset of this lane's sector inside the row
                    if (((wv >> lane) & 1u) && off < row_bytes) {
                        o[u] = f * frame_stride + (int64_t)row * row_stride + off;
                        nb[u] = min(32, row_bytes - off);
                    }
                }
            }
            uint4 va[4], vb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (nb[u] >= 16) va[u] = __ldcs(reinterpret_cast<const uint4*>(src + o[u]));
                if (nb[u] >= 32) vb[u] = __ldcs(reinterpret_cast<const uint4*>(src + o[u] + 16));
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (nb[u] >= 16) *reinterpret_cast<uint4*>(mirror + o[u]) = va[u];
                if (nb[u] >= 32) *reinterpret_cast<uint4*>(mirror + o[u] + 16) = vb[u];
                copied += (unsigned)(nb[u] & ~15);
            }
        }
    }
    copied = warp_sum_u64(copied);
    if (lane == 0 && copied && bytes_out) atomicAdd(bytes_out, copied);
}

// =====================================================================================================
// K3  getColorMaskRedOrBlue(img,'r'/'b')  (DET:63-89), SURVEY A.3.  One thread per pixel; integer HSV tables.
// `slots` (optional) = indirection to the surviving windows inside the work buffer.
// =====================================================================================================
// K3 v2: one warp per window, lane-strided pixels (coalesced byte loads, stride 3), mask bytes written with stride `ms`
// (npx for the public packed layout, padded to 16 for the internal one) and, optionally, the same masks bit-packed
// (pixel p -> word p>>5, bit p&31; [w][0..NW) red, [w][NW..2NW) blue) which is what K4 consumes inside the chain.
__global__ void __launch_bounds__(256) k3_masks_generic_kernel(const uint8_t* __restrict__ windows, const int32_t* __restrict__ slots,
                                                          const int32_t* __restrict__ n_ptr, int n_max, int npx, int ws,
                                                          const Tables* __restrict__ tab, HsvBounds hb, uint8_t* __restrict__ red,
                                                          uint8_t* __restrict__ blue, int ms, uint32_t* __restrict__ bits) {
    __shared__ int32_t s_sdiv[256], s_hdiv[256];
    s_sdiv[threadIdx.x & 255] = tab->sdiv[threadIdx.x & 255];
    s_hdiv[threadIdx.x & 255] = tab->hdiv[threadIdx.x & 255];
    __syncthreads();
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int lane = threadIdx.x & 31, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int NW = (npx + 31) >> 5;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += nwarps) {
        const uint8_t* __restrict__ px = windows + (int64_t)(slots ? slots[w] : w) * ws;
        uint8_t* __restrict__ ro = red + (int64_t)w * ms;
        uint8_t* __restrict__ bo = blue + (int64_t)w * ms;
        uint32_t myr = 0, myb = 0;
#pragma unroll 4
        for (int i = 0; i < NW; i++) {
            const int p = i * 32 + lane;
            const bool valid = p < npx;
            const int pp = valid ? p : 0;
            const int b = __ldg(px + 3 * pp), g = __ldg(px + 3 * pp + 1), r = __ldg(px + 3 * pp + 2);
            int H, S, V;
            bgr2hsv(b, g, r, s_sdiv, s_hdiv, H, S, V);
            const bool r0 = H >= hb.red_lo[0][0] && H <= hb.red_hi[0][0] && S >= hb.red_lo[0][1] && S <= hb.red_hi[0][1] &&
                            V >= hb.red_lo[0][2] && V <= hb.red_hi[0][2];
            const bool r1 = H >= hb.red_lo[1][0] && H <= hb.red_hi[1][0] && S >= hb.red_lo[1][1] && S <= hb.red_hi[1][1] &&
                            V >= hb.red_lo[1][2] && V <= hb.red_hi[1][2];
            const bool bl = H >= hb.blue_lo[0] && H <= hb.blue_hi[0] && S >= hb.blue_lo[1] && S <= hb.blue_hi[1] &&
                            V >= hb.blue_lo[2] && V <= hb.blue_hi[2];
            const bool rr = r0 || r1;                       // cv2.add of the two bands saturates at 255
            if (valid) { ro[p] = rr ? 255 : 0; bo[p] = bl ? 255 : 0; }
            const unsigned wr = __ballot_sync(0xffffffffu, valid && rr), wb = __ballot_sync(0xffffffffu, valid && bl);
            if (lane == i) { myr = wr; myb = wb; }
        }
        if (bits && lane < NW) { bits[(int64_t)w * 2 * NW + lane] = myr; bits[(int64_t)w * 2 * NW + NW + lane] = myb; }
    }
}

// K3 v3 (internal layout only): v2 + (1) the inRange tests become three byte-table lookups AND-ed together (bit 0/1 = the two
// red bands, bit 2 = blue; tables built on the host from tsd_config, so any bounds work), (2) the next window travels into
// registers with 128-bit loads while the current one is processed from shared memory (v2 stalled on its byte loads).
struct MaskLut { uint8_t hf[256], sf[256], vf[256]; };

template <int NCH>
__global__ void __launch_bounds__(256) k3_masks_v3_kernel(const uint8_t* __restrict__ windows, const int32_t* __restrict__ slots,
                                                          const int32_t* __restrict__ n_ptr, int n_max, int npx, int ws,
                                                          const Tables* __restrict__ tab, const MaskLut* __restrict__ mlut,
                                                          uint8_t* __restrict__ red, uint8_t* __restrict__ blue, int ms, uint32_t* __restrict__ bits) {
    __shared__ int32_t s_sdiv[256], s_hdiv[256];
    __shared__ uint8_t s_hf[256], s_sf[256], s_vf[256];
    __shared__ uint4 s_px[8][NCH * 32];
    s_sdiv[threadIdx.x & 255] = tab->sdiv[threadIdx.x & 255];
    s_hdiv[threadIdx.x & 255] = tab->hdiv[threadIdx.x & 255];
    s_hf[threadIdx.x & 255] = mlut->hf[threadIdx.x & 255];
    s_sf[threadIdx.x & 255] = mlut->sf[threadIdx.x & 255];
    s_vf[threadIdx.x & 255] = mlut->vf[threadIdx.x & 255];
    __syncthreads();
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int NW = (npx + 31) >> 5, nch = ws >> 4;
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint4 r[NCH];
    int slot_next = 0;                                       // slot of window w + nwarps (loaded one iteration ahead)
    if (w < n) {
        const int s0 = slots ? __ldg(slots + w) : w;
        const uint4* g = reinterpret_cast<const uint4*>(windows + (int64_t)s0 * ws);
#pragma unroll
        for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) r[k] = __ldg(g + lane + 32 * k);
        if (w + nwarps < n) slot_next = slots ? __ldg(slots + w + nwarps) : w + nwarps;
    }
    const uint8_t* px = reinterpret_cast<const uint8_t*>(s_px[wid]);
    for (; w < n; w += nwarps) {
#pragma unroll
        for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) s_px[wid][lane + 32 * k] = r[k];
        __syncwarp();
        if (w + nwarps < n) {
            const uint4* g = reinterpret_cast<const uint4*>(windows + (int64_t)slot_next * ws);
#pragma unroll
            for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) r[k] = __ldg(g + lane + 32 * k);
            if (w + 2 * nwarps < n) slot_next = slots ? __ldg(slots + w + 2 * nwarps) : w + 2 * nwarps;
        }
        uint8_t* __restrict__ ro = red + (int64_t)w * ms;
        uint8_t* __restrict__ bo = blue + (int64_t)w * ms;
        uint32_t myr = 0, myb = 0;
#pragma unroll kK3Unroll
        for (int i = 0; i < NW; i++) {
            const int p = i * 32 + lane;
            const bool valid = p < npx;
            const int pp = valid ? p : 0;
            const int b = px[3 * pp], g = px[3 * pp + 1], rr = px[3 * pp + 2];
            int H, S, V;
            bgr2hsv(b, g, rr, s_sdiv, s_hdiv, H, S, V);
            const unsigned fl = valid ? (unsigned)(s_hf[H] & s_sf[S] & s_vf[V]) : 0u;
            if (valid && red) { ro[p] = (fl & 3u) ? 255 : 0; bo[p] = (fl & 4u) ? 255 : 0; }     // cv2.add of the two red bands saturates at 255
            const unsigned wr = __ballot_sync(0xffffffffu, (fl & 3u) != 0), wb = __ballot_sync(0xffffffffu, (fl & 4u) != 0);
            if (lane == i) { myr = wr; myb = wb; }
        }
        if (bits && lane < NW) { bits[(int64_t)w * 2 * NW + lane] = myr; bits[(int64_t)w * 2 * NW + NW + lane] = myb; }
        __syncwarp();                                        // all taps read before the staging buffer is overwritten
    }
}

__global__ void bgr2hsv_kernel(const uint8_t* __restrict__ bgr, int64_t npx, const Tables* __restrict__ tab,
                               uint8_t* __restrict__ hsv) {
    __shared__ int32_t s_sdiv[256], s_hdiv[256];
    s_sdiv[threadIdx.x & 255] = tab->sdiv[threadIdx.x & 255];
    s_hdiv[threadIdx.x & 255] = tab->hdiv[threadIdx.x & 255];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (int64_t)gridDim.x * blockDim.x) {
        int H, S, V;
        bgr2hsv(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2], s_sdiv, s_hdiv, H, S, V);
        hsv[3 * i] = (uint8_t)H; hsv[3 * i + 1] = (uint8_t)S; hsv[3 * i + 2] = (uint8_t)V;
    }
}

// =====================================================================================================
// K4  getSimilarSignalType x2 + detectionsMaskCorrelation decision  (DET:229-261,545-567), SURVEY A.4.
// mask*template wraps to {0,1} so FP == 0, FN = T - TP, TN = npx - T: the score depends on (TP, template) only.
// Templates are bit-packed (32 px / word); lut[k][TP] = hundredths of round(2TP/(TP+T_k), 2) or 0 when the
// template is degenerate -- built on the host with the reference's own arithmetic.
// One warp per window: 32 mask bytes -> one ballot word; lane k < 12 accumulates popc(word & template_k).
// =====================================================================================================
struct ScoreTemplates {
    uint32_t bits[12][kMaxPx / 32];      // [0..5] red, [6..11] blue
    uint8_t lut[12][kMaxPx + 1];
};

__global__ void __launch_bounds__(128) k4_score_kernel(const uint8_t* __restrict__ red, const uint8_t* __restrict__ blue,
                                                       const int32_t* __restrict__ n_ptr, int n_max, int npx, int ms,
                                                       const ScoreTemplates* __restrict__ tmpl, int tol_hundredths,
                                                       int32_t* __restrict__ scores, int32_t* __restrict__ id,
                                                       int32_t* __restrict__ hundredths, uint8_t* __restrict__ emit) {
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    if (w >= n) return;
    const uint8_t* r = red + (int64_t)w * ms;
    const uint8_t* b = blue + (int64_t)w * ms;
    const int nwords = (npx + 31) >> 5;
    int tp = 0;
    for (int i = 0; i < nwords; i++) {
        int p = i * 32 + lane;
        unsigned wr = __ballot_sync(0xffffffffu, p < npx && r[p] != 0);
        unsigned wb = __ballot_sync(0xffffffffu, p < npx && b[p] != 0);
        if (lane < 12) tp += __popc((lane < 6 ? wr : wb) & tmpl->bits[lane][i]);
    }
    int sc = lane < 12 ? (int)tmpl->lut[lane][tp] : -1;
    if (scores && lane < 12) scores[(int64_t)w * 12 + lane] = sc;
    // first strict maximum within each group of 6 (DET:249-259)
    int best_r = -1, id_r = 0, best_b = -1, id_b = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        int sr = __shfl_sync(0xffffffffu, sc, k), sb = __shfl_sync(0xffffffffu, sc, 6 + k);
        if (sr > best_r) { best_r = sr; id_r = k + 1; }
        if (sb > best_b) { best_b = sb; id_b = k + 1; }
    }
    if (lane == 0) {
        bool red_wins = best_r > best_b;                    // tie -> blue (DET:236)
        int s = red_wins ? best_r : best_b;
        id[w] = red_wins ? id_r : id_b;
        hundredths[w] = s;
        emit[w] = s > tol_hundredths ? 1 : 0;
    }
}

// K4 v2 (inside the chain): the same decision from K3's bit-packed masks.  One THREAD per window: 2*NW mask words in
// registers (128-bit loads), 12 x NW template words in shared memory (broadcast reads), popcounts, LUT, decision.
template <int NW>
__global__ void __launch_bounds__(128) k4_score_bits_kernel(const uint32_t* __restrict__ bits, const int32_t* __restrict__ n_ptr, int n_max,
                                                            const ScoreTemplates* __restrict__ tmpl, int tol_hundredths,
                                                            int32_t* __restrict__ id, int32_t* __restrict__ hundredths, uint8_t* __restrict__ emit) {
    __shared__ uint32_t s_t[12][NW];
    for (int i = threadIdx.x; i < 12 * NW; i += blockDim.x) s_t[i / NW][i % NW] = tmpl->bits[i / NW][i % NW];
    __syncthreads();
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n) return;
    static_assert(NW % 4 == 0, "mask words are loaded 4 at a time");
    const uint4* src = reinterpret_cast<const uint4*>(bits + (int64_t)w * 2 * NW);
    int tp[12];
#pragma unroll
    for (int k = 0; k < 12; k++) tp[k] = 0;
#pragma unroll
    for (int q = 0; q < NW / 4; q++) {
        const uint4 vr = __ldg(src + q), vb = __ldg(src + NW / 4 + q);
        const uint32_t wr[4] = {vr.x, vr.y, vr.z, vr.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int k = 0; k < 6; k++) {
                tp[k] += __popc(wr[u] & s_t[k][4 * q + u]);
                tp[6 + k] += __popc(wb[u] & s_t[6 + k][4 * q + u]);
            }
        }
    }
    // first strict maximum within each group of 6 (DET:249-259); red wins only if strictly better (DET:236)
    int best_r = -1, id_r = 0, best_b = -1, id_b = 0;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const int sr = (int)__ldg(&tmpl->lut[k][tp[k]]), sb = (int)__ldg(&tmpl->lut[6 + k][tp[6 + k]]);
        if (sr > best_r) { best_r = sr; id_r = k + 1; }
        if (sb > best_b) { best_b = sb; id_b = k + 1; }
    }
    const bool red_wins = best_r > best_b;
    const int sc = red_wins ? best_r : best_b;
    id[w] = red_wins ? id_r : id_b;
    hundredths[w] = sc;
    emit[w] = sc > tol_hundredths ? 1 : 0;
}

// =====================================================================================================
// K5  cleanDuplicatedDetections (DET:177-223) -- SURVEY A.5.
// Per-window sparse H-S histogram record (calculateHistAndNormalize DET:575-586):
//   entries (bin << 16 | count), sorted by bin; a = (float)(1/max) ; h[bin] = (float)count * a  (min is always 0
//   because npx <= 1024 < 3000 bins, so the MINMAX shift is +0);  s1 = sum h, s11 = sum h^2 in f64;
//   hash = 32-bit order-independent hash of the pixels (pix_hash32 sum; only pre-filters the pop-by-pixel-equality rule DET:471-477).
// =====================================================================================================
struct __align__(16) WinMeta {
    double s1, s11;              // sum h, sum h^2 over the 3000 bins (f64)
    double A, rA;                // A = s11 - s1*s1/N (one factor of compareHist's denom2), rA = sqrt(A)
    float a;                     // (float)(1/max count)
    int32_t nnz;
    uint32_t hash;               // pix_hash32 sum
    uint32_t pad_;
};
static_assert(sizeof(WinMeta) == 48, "WinMeta layout");

__device__ __forceinline__ uint32_t warp_sum_u(uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide: histogram of one window.  dense[kHistBins] (shared, zero on entry, left holding the counts),
// red[] = shared scratch of >= 64 doubles.  Writes entries + meta for `slot`.  All threads must call.
__device__ void build_hist_block(const uint8_t* __restrict__ px, int npx, const int32_t* s_sdiv, const int32_t* s_hdiv,
                                 const uint8_t* s_hbin, const uint8_t* s_sbin, uint32_t* dense, double* red,
                                 uint32_t* __restrict__ entries, WinMeta* __restrict__ meta) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    uint32_t hsh = 0;
    for (int p = tid; p < npx; p += nt) {
        int b = px[3 * p], g = px[3 * p + 1], r = px[3 * p + 2];
        int H, S, V;
        bgr2hsv(b, g, r, s_sdiv, s_hdiv, H, S, V);
        atomicAdd(&dense[(int)s_hbin[H] * kHistS + (int)s_sbin[S]], 1u);
        hsh += pix_hash32(p, (uint32_t)(b | (g << 8) | (r << 16)));
    }
    hsh = warp_sum_u(hsh);                                  // order-independent sum of per-pixel mixes
    uint32_t* red_u = reinterpret_cast<uint32_t*>(red);
    __syncthreads();
    if (lane == 0) red_u[wid] = hsh;
    __syncthreads();
    uint32_t hash_all = 0;
    for (int i = 0; i < nw; i++) hash_all += red_u[i];
    __syncthreads();
    // max count + per-warp nnz over contiguous bin ranges (deterministic, sorted-by-bin output)
    const int per_warp = (kHistBins + nw - 1) / nw;
    const int b0 = wid * per_warp, b1 = min(kHistBins, b0 + per_warp);
    unsigned mx = 0; int cnt = 0;
    for (int b = b0 + lane; b < b1; b += 32) { unsigned c = dense[b]; mx = max(mx, c); cnt += c != 0; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o)); cnt += __shfl_xor_sync(0xffffffffu, cnt, o); }
    int* red_i = reinterpret_cast<int*>(red);
    if (lane == 0) { red_i[wid] = (int)mx; red_i[32 + wid] = cnt; }
    __syncthreads();
    unsigned mx_all = 0; int base = 0, nnz = 0;
    for (int i = 0; i < nw; i++) { mx_all = max(mx_all, (unsigned)red_i[i]); if (i < wid) base += red_i[32 + i]; nnz += red_i[32 + i]; }
    __syncthreads();
    // normalize: scale = 1/(max-min) in f64, a = (float)scale (cv2.normalize NORM_MINMAX -> convertTo)
    double scale = ((double)mx_all - 0.0) > DBL_EPSILON ? 1.0 / ((double)mx_all - 0.0) : 0.0;
    float a = (float)scale;
    double s1 = 0, s11 = 0;
    int outp = base;
    for (int bb = b0; bb < b1; bb += 32) {
        int b = bb + lane;
        unsigned c = b < b1 ? dense[b] : 0;
        unsigned m = __ballot_sync(0xffffffffu, c != 0);
        if (c) {
            entries[outp + __popc(m & ((1u << lane) - 1))] = ((uint32_t)b << 16) | c;
            double h = (double)((float)c * a);
            s1 += h; s11 += h * h;
        }
        outp += __popc(m);
    }
    s1 = warp_sum(s1); s11 = warp_sum(s11);
    if (lane == 0) { red[wid] = s1; red[32 + wid] = s11; }
    __syncthreads();
    if (tid == 0) {
        double t1 = 0, t11 = 0;
        for (int i = 0; i < nw; i++) { t1 += red[i]; t11 += red[32 + i]; }
        const double A = t11 - t1 * t1 * (1.0 / (double)kHistBins);
        meta->s1 = t1; meta->s11 = t11; meta->A = A; meta->rA = sqrt(A); meta->hash = hash_all; meta->a = a; meta->nnz = nnz; meta->pad_ = 0;
    }
    __syncthreads();
}

// zero the dense histogram entries listed in `entries` (cheaper than clearing all 3000 bins)
__device__ __forceinline__ void clear_dense_block(uint32_t* dense, const uint32_t* __restrict__ entries, int nnz) {
    for (int e = threadIdx.x; e < nnz; e += blockDim.x) dense[entries[e] >> 16] = 0;
}

struct HistSmem {
    int32_t sdiv[256], hdiv[256];
    uint8_t hbin[256], sbin[256];
    uint32_t dense[kHistBins];
    double red[64];
};

__device__ __forceinline__ void load_tables_block(HistSmem& sm, const Tables* __restrict__ tab) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sm.sdiv[i] = tab->sdiv[i]; sm.hdiv[i] = tab->hdiv[i]; sm.hbin[i] = tab->hbin[i]; sm.sbin[i] = tab->sbin[i];
    }
    for (int i = threadIdx.x; i < kHistBins; i += blockDim.x) sm.dense[i] = 0;
}

// dense float32 [n][50][60] normalised histograms (tsd_hist, parity artefact of calculateHistAndNormalize)
__global__ void hist_dense_kernel(const uint32_t* __restrict__ entries, const WinMeta* __restrict__ meta, int n, int es,
                                  float* __restrict__ out) {
    int w = blockIdx.x;
    if (w >= n) return;
    float* o = out + (int64_t)w * kHistBins;
    for (int i = threadIdx.x; i < kHistBins; i += blockDim.x) o[i] = 0.f;
    __syncthreads();
    const uint32_t* e = entries + (int64_t)w * es;
    float a = meta[w].a;
    for (int i = threadIdx.x; i < meta[w].nnz; i += blockDim.x) o[e[i] >> 16] = (float)(e[i] & 0xffffu) * a;
}

// pixel hash only (pass-2-only entry point): one warp per window
__global__ void __launch_bounds__(128) k5_hash_kernel(const uint8_t* __restrict__ windows, int n, int npx, int ws, WinMeta* __restrict__ meta) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const uint8_t* px = windows + (int64_t)w * ws;
    uint32_t hsh = 0;
    for (int p = lane; p < npx; p += 32) hsh += pix_hash32(p, (uint32_t)(px[3 * p] | (px[3 * p + 1] << 8) | (px[3 * p + 2] << 16)));
    hsh = warp_sum_u(hsh);
    if (lane == 0) meta[w].hash = hsh;
}

// ---- the fold ----------------------------------------------------------------------------------------
struct FoldParams {
    uint8_t* windows;            // work buffer [n][npx*3]; merged items are averaged IN PLACE in the item's slot
    int4* coords;                // [n]; merged coords are written in place
    uint32_t* entries;           // [n][npx] sparse histograms
    WinMeta* meta;               // [n]
    const int32_t* offsets;      // [nframes+1] CSR of the input windows
    int32_t* list;               // [n] scratch: per frame, list positions -> slot (frame's region = its CSR range)
    uint8_t* flags;              // [n] scratch: deletion marks per list position
    int32_t* out_count;          // [nframes] survivors per frame
    const double* simtab;        // f(d2), d2 < simtab_n (DET:459-462)
    int simtab_n;
    const Tables* tab;
    int npx, ws, es;             // pixels per window; window stride (bytes); entry stride (words)
    float* E_T;                  // group energies [25][e_stride] of the windows (pruning bound; rewritten for merged items), NULL when !do_hist
    int64_t e_stride;
    int do_hist, do_coords;      // which passes to run (DET:127 then DET:129)
    double hist_tol, hist_lo, coord_tol, coord_lo;   // lo = tol * 0.8823 (DET:217), computed on the host in f64
};

constexpr int kFoldThreads = 256;
constexpr int kFoldChunk = 1024;

struct FoldSmem {
    HistSmem h;
    uint8_t cls[kFoldChunk];
    int first_merge;
    int any_del;
    int S;
    int4 icoords;
    int victim;
};

__device__ __forceinline__ double coord_sim(int4 a, int4 b, const double* __restrict__ simtab, int simtab_n) {
    // 32-bit arithmetic: a corner more than 32767 px away in x or y is beyond every table (simtab_n <= 2^30) without squaring it
    const int dx = a.x - b.x, dy = a.y - b.y, ex = a.z - b.z, ey = a.w - b.w;
    if (max(max(abs(dx), abs(dy)), max(abs(ex), abs(ey))) > 32767) return 0.0;
    const int d1 = dx * dx + dy * dy, d2 = ex * ex + ey * ey;
    // beyond the table f(d) <= f(simtab_n - 1), and the host refuses a tolerance unless sqrt(f(simtab_n - 1)) < tol * merge_factor
    // (check_simtab): such a pair takes no action, as in the reference
    if (d1 >= simtab_n || d2 >= simtab_n) return 0.0;
    return __dsqrt_rn(__dmul_rn(simtab[d1], simtab[d2]));
}

// pop-by-pixel-equality (DET:183-185,471-477): for each marked position, in list order, remove the FIRST live entry
// whose pixels equal the marked one's.  Then compact the list.  Block-wide; returns the new length in sm.S.
__device__ void apply_deletions_block(FoldSmem& sm, const FoldParams& P, int32_t* list, uint8_t* flags, int nbytes) {
    const int tid = threadIdx.x;
    const int S = sm.S;
    // flags: 1 = marked for deletion (by scan), 2 = dead (already removed).  Process marks in increasing position.
    for (int p = 0; p < S; p++) {
        if (flags[p] != 1) continue;                        // uniform across the block (global memory, synced)
        const int slot_d = list[p];
        const uint32_t hd = P.meta[slot_d].hash;
        if (tid == 0) sm.victim = p;
        __syncthreads();
        // earlier live entries (flag 0 or 1) with equal hash -> verify bytes; smallest position wins
        for (int q = tid; q < p; q += blockDim.x) {
            if (flags[q] != 2 && P.meta[list[q]].hash == hd) {
                const uint8_t* A = P.windows + (int64_t)list[q] * P.ws;
                const uint8_t* B = P.windows + (int64_t)slot_d * P.ws;
                bool eq = true;
                for (int i = 0; i < nbytes; i++) if (A[i] != B[i]) { eq = false; break; }
                if (eq) atomicMin(&sm.victim, q);
            }
        }
        __syncthreads();
        const int v = sm.victim;
        __syncthreads();
        if (tid == 0) {
            // the victim leaves the list; if it was itself marked, that mark is consumed with it and the entry at p
            // stays pending only if v != p -- in the reference the second pop then removes the next equal entry,
            // which is p itself once v is gone (v's own mark, processed earlier, cannot exist since v < p was live+unprocessed
            // only if unmarked or marked-later; marks are processed in order, so a marked v < p was already handled).
            flags[v] = 2;
            if (v != p) flags[p] = 0;                       // p survives (its twin was popped instead)
        }
        __syncthreads();
    }
    // compaction by warp 0, order preserving
    if (tid < 32) {
        int outp = 0;
        for (int base = 0; base < S; base += 32) {
            int p = base + tid;
            bool live = p < S && flags[p] != 2;
            int slot = p < S ? list[p] : 0;
            unsigned m = __ballot_sync(0xffffffffu, live);
            __syncwarp();
            if (live) list[outp + __popc(m & ((1u << tid) - 1))] = slot;
            outp += __popc(m);
            __syncwarp();
        }
        if (tid == 0) sm.S = outp;
    }
    __syncthreads();
    for (int p = tid; p < S; p += blockDim.x) flags[p] = 0;
    __syncthreads();
}

// One CTA per frame.  Sequential over the frame's items (the fold order is the semantics); each item is compared
// with ALL current survivors in parallel, the classes are scanned in list order up to the first merge, the merge is
// applied and only the survivors after it are re-evaluated with the updated item (speculate-then-scan).
// surv_offsets (optional): the last CTA to finish turns out_count [nframes] (written by this kernel and by the per-warp / per-CTA
// folds launched before it) into the CSR offsets of the survivors.
__global__ void __launch_bounds__(kFoldThreads) k5_fold_kernel(FoldParams P, int nframes, int only_flagged, int32_t* __restrict__ surv_offsets,
                                                               unsigned* __restrict__ ticket) {
    __shared__ FoldSmem sm;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = kFoldThreads >> 5;
    const int nbytes = P.npx * 3;
    if (P.do_hist) load_tables_block(sm.h, P.tab);
    if (tid == 0) sm.any_del = 0;
    __syncthreads();
    for (int f = blockIdx.x; f < nframes; f += gridDim.x) {
        if (only_flagged && P.out_count[f] != -1) continue;  // the warp-per-frame fold already did this frame (block-uniform)
        const int base = P.offsets[f], n = P.offsets[f + 1] - base;
        int32_t* list = P.list + base;
        uint8_t* flags = P.flags + base;
        for (int p = tid; p < n; p += blockDim.x) flags[p] = 0;
        if (tid == 0) sm.S = 0;
        __syncthreads();
        for (int pass = 0; pass < 2; pass++) {
            const bool by_coords = pass == 1;
            if (by_coords ? !P.do_coords : !P.do_hist) continue;
            const double tol = by_coords ? P.coord_tol : P.hist_tol, lo = by_coords ? P.coord_lo : P.hist_lo;
            // items of this pass: pass 0 (or coords-only) -> slots base..base+n-1 in order; pass 1 after pass 0 -> the
            // survivors of pass 0, which we first move aside to the tail of the scratch region as the "input" order.
            // To avoid a second array the input order is read from `list` itself: survivors of pass 0 occupy
            // list[0..S0) and pass 1 rebuilds the list in place (the write index never passes the read index).
            const bool from_list = by_coords && P.do_hist;
            const int nin = from_list ? sm.S : n;
            __syncthreads();
            if (tid == 0) sm.S = 0;
            __syncthreads();
            for (int it = 0; it < nin; it++) {
                const int slot = from_list ? list[it] : base + it;
                __syncthreads();                            // list[it] read before anyone overwrites it below
                uint8_t* ipx = P.windows + (int64_t)slot * P.ws;
                uint32_t* ient = P.entries + (int64_t)slot * P.es;
                if (tid == 0) sm.icoords = P.coords[slot];
                if (!by_coords) {
                    const int nnz = P.meta[slot].nnz;
                    for (int e = tid; e < nnz; e += blockDim.x) { uint32_t v = ient[e]; sm.h.dense[v >> 16] = v & 0xffffu; }
                }
                __syncthreads();
                int start = 0;
                while (start < sm.S) {
                    const int S = sm.S;
                    const int end = min(S, start + kFoldChunk);
                    if (tid == 0) sm.first_merge = 0x7fffffff;
                    __syncthreads();
                    if (by_coords) {
                        const int4 ic = sm.icoords;
                        for (int p = start + tid; p < end; p += blockDim.x) {
                            double sim = coord_sim(ic, P.coords[list[p]], P.simtab, P.simtab_n);
                            int c = sim > tol ? 1 : (lo <= sim && sim <= tol) ? 2 : 0;
                            sm.cls[p - start] = (uint8_t)c;
                            if (c == 2) atomicMin(&sm.first_merge, p);
                        }
                    } else {
                        const WinMeta mi = P.meta[slot];
                        for (int p = start + wid; p < end; p += nw) {
                            const int sj = list[p];
                            const WinMeta mj = P.meta[sj];
                            const uint32_t* ej = P.entries + (int64_t)sj * P.es;
                            double s12 = 0;
                            for (int e = lane; e < mj.nnz; e += 32) {
                                uint32_t v = ej[e];
                                float hi = (float)sm.h.dense[v >> 16] * mi.a;
                                float hj = (float)(v & 0xffffu) * mj.a;
                                s12 += (double)hi * (double)hj;
                            }
                            s12 = warp_sum(s12);
                            if (lane == 0) {
                                // cv2.compareHist CORREL (DET:200-202): h1 = item, h2 = survivor
                                const double scale = 1.0 / (double)kHistBins;
                                double num = s12 - mi.s1 * mj.s1 * scale;
                                double den2 = (mi.s11 - mi.s1 * mi.s1 * scale) * (mj.s11 - mj.s1 * mj.s1 * scale);
                                double sim = fabs(den2) > DBL_EPSILON ? num / sqrt(den2) : 1.0;
                                int c = sim > tol ? 1 : (lo <= sim && sim <= tol) ? 2 : 0;
                                sm.cls[p - start] = (uint8_t)c;
                                if (c == 2) atomicMin(&sm.first_merge, p);
                            }
                        }
                    }
                    __syncthreads();
                    const int fm = sm.first_merge;
                    const int lim = min(fm, end);
                    for (int p = start + tid; p < lim; p += blockDim.x)
                        if (sm.cls[p - start] == 1) { flags[p] = 1; sm.any_del = 1; }
                    if (fm < end) {
                        // merge (DET:217-221): pixels = addWeighted(.5,.5) round-half-even, coords = floor mean
                        const int sk = list[fm];
                        const uint8_t* kpx = P.windows + (int64_t)sk * P.ws;
                        if (!by_coords) clear_dense_block(sm.h.dense, ient, P.meta[slot].nnz);
                        for (int i = tid; i < nbytes; i += blockDim.x) {
                            int s = ipx[i] + kpx[i];
                            ipx[i] = (uint8_t)((s >> 1) + ((s & 1) & ((s >> 1) & 1)));
                        }
                        if (tid == 0) {
                            int4 a = sm.icoords, b = P.coords[sk];
                            // Python // on ints (coords are >= 0)
                            sm.icoords = make_int4((a.x + b.x) >> 1, (a.y + b.y) >> 1, (a.z + b.z) >> 1, (a.w + b.w) >> 1);
                            flags[fm] = 1; sm.any_del = 1;
                        }
                        __syncthreads();
                        if (!by_coords) {
                            build_hist_block(ipx, P.npx, sm.h.sdiv, sm.h.hdiv, sm.h.hbin, sm.h.sbin, sm.h.dense, sm.h.red, ient, P.meta + slot);
                        } else {
                            // keep the pixel hash current for the pop-by-equality rule
                            uint32_t hsh = 0;
                            for (int p = tid; p < P.npx; p += blockDim.x)
                                hsh += pix_hash32(p, (uint32_t)(ipx[3 * p] | (ipx[3 * p + 1] << 8) | (ipx[3 * p + 2] << 16)));
                            hsh = warp_sum_u(hsh);
                            uint32_t* ru = reinterpret_cast<uint32_t*>(sm.h.red);
                            if (lane == 0) ru[wid] = hsh;
                            __syncthreads();
                            if (tid == 0) { uint32_t t = 0; for (int i = 0; i < nw; i++) t += ru[i]; P.meta[slot].hash = t; }
                            __syncthreads();
                        }
                        start = fm + 1;
                    } else {
                        start = end;
                    }
                    __syncthreads();
                }
                __syncthreads();
                if (!by_coords) clear_dense_block(sm.h.dense, ient, P.meta[slot].nnz);
                if (tid == 0) P.coords[slot] = sm.icoords;
                __syncthreads();
                if (sm.any_del) {
                    apply_deletions_block(sm, P, list, flags, nbytes);
                    if (tid == 0) sm.any_del = 0;
                }
                __syncthreads();
                if (tid == 0) { list[sm.S] = slot; sm.S = sm.S + 1; }
                __syncthreads();
            }
        }
        __syncthreads();
        if (!(P.do_hist || P.do_coords)) {                  // no pass requested: identity
            for (int p = tid; p < n; p += blockDim.x) list[p] = base + p;
            if (tid == 0) sm.S = n;
            __syncthreads();
        }
        if (tid == 0) P.out_count[f] = sm.S;
        __syncthreads();
    }
    if (surv_offsets) scan_by_last_block(P.out_count, nframes, surv_offsets, ticket);
}

// gather survivors (list -> compact CSR output).  One CTA per frame.
__global__ void k5_gather_kernel(const uint8_t* __restrict__ windows, const int4* __restrict__ coords,
                                 const int32_t* __restrict__ in_offsets, const int32_t* __restrict__ list,
                                 const int32_t* __restrict__ out_offsets, int nframes, int nbytes, int ws,
                                 uint8_t* __restrict__ out_windows, int4* __restrict__ out_coords, int32_t* __restrict__ out_slots) {
    int f = blockIdx.x;
    if (f >= nframes) return;
    const int o0 = out_offsets[f], cnt = out_offsets[f + 1] - o0;
    const int32_t* l = list + in_offsets[f];
    for (int r = 0; r < cnt; r++) {
        const int slot = l[r];
        if (out_windows) {
            const uint8_t* s = windows + (int64_t)slot * ws;
            uint8_t* d = out_windows + (int64_t)(o0 + r) * nbytes;     // public layout: packed
            for (int i = threadIdx.x; i < nbytes; i += blockDim.x) d[i] = s[i];
        }
        if (threadIdx.x == 0) {
            if (out_coords) out_coords[o0 + r] = coords[slot];
            if (out_slots) out_slots[o0 + r] = slot;
        }
    }
}

// =====================================================================================================
// K6  cv2.cvtColor(BGR2GRAY)  (REC:388), SURVEY A.6
// =====================================================================================================
__global__ void k6_gray_kernel(const uint8_t* __restrict__ windows, const int32_t* __restrict__ slots,
                               const int32_t* __restrict__ n_ptr, int n_max, int npx, int ws, uint8_t* __restrict__ gray) {
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int64_t total = (int64_t)n * npx;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int w = (int)(i / npx);
        const uint8_t* p = windows + (int64_t)(slots ? slots[w] : w) * ws + (i - (int64_t)w * npx) * 3;
        gray[i] = (uint8_t)((3735 * p[0] + 19235 * p[1] + 9798 * p[2] + 16384) >> 15);
    }
}

// =====================================================================================================
// N1  grayAndEnhanceContrast (DET:135-152 = REC:67-84): BGR2GRAY -> CLAHE(clip 2, 8x8 tiles) -> GaussianBlur 3x3 -> gamma LUT.
// The proposal pre-processing that feeds cv2.MSER (SURVEY 8(f) N1).  Two kernels:
//   pre_gray_lut   : one CTA per (tile, frame): grey conversion of the tile (written out), its 256-bin histogram in shared
//                    memory, clip + redistribution + cumulative sum -> the tile's 256-entry LUT (OpenCV clahe.cpp, including
//                    the BORDER_REFLECT_101 extension of images that are not a multiple of the grid).
//   pre_clahe_blur : one CTA per 64x16 output pixels: the CLAHE value (float bilinear blend of 4 tile LUTs, OpenCV's exact
//                    operation order, no FMA) of the tile + 1-pixel halo into shared memory, then the exact (1 2 1)x(1 2 1)/16
//                    blur with round-half-up and the gamma table.
// =====================================================================================================
__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i;
    return i;
}

__global__ void __launch_bounds__(256) pre_gray_lut_kernel(const uint8_t* __restrict__ frames, int H, int W, int64_t row_stride, int64_t frame_stride,
                                                           int tiles_x, int tiles_y, int tw, int th, int clip, float lut_scale,
                                                           uint8_t* __restrict__ gray, uint8_t* __restrict__ luts) {
    __shared__ int s_hist[256];
    __shared__ int s_part[8];
    const int tile = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const uint8_t* __restrict__ fr = frames + (int64_t)f * frame_stride;
    uint8_t* __restrict__ go = gray + (int64_t)f * H * W;
    s_hist[tid] = 0;
    __syncthreads();
    for (int r = wid; r < th; r += 8) {
        const int ye = ty * th + r, y = reflect101(ye, H);
        const uint8_t* __restrict__ row = fr + (int64_t)y * row_stride;
        for (int cidx = lane; cidx < tw; cidx += 32) {
            const int xe = tx * tw + cidx, x = reflect101(xe, W);
            const int g = (3735 * __ldg(row + 3 * x) + 19235 * __ldg(row + 3 * x + 1) + 9798 * __ldg(row + 3 * x + 2) + 16384) >> 15;   // A.6
            atomicAdd(&s_hist[g], 1);
            if (ye < H && xe < W) go[(int64_t)ye * W + xe] = (uint8_t)g;
        }
    }
    __syncthreads();
    int h = s_hist[tid];
    if (clip > 0) {
        int excess = h > clip ? h - clip : 0;
        h = h > clip ? clip : h;
        int e = warp_sum_i(excess);
        if (lane == 0) s_part[wid] = e;
        __syncthreads();
        int clipped = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) clipped += s_part[k];
        const int batch = clipped >> 8, residual = clipped - (batch << 8);
        h += batch;
        if (residual != 0) {
            int step = 256 / residual; if (step < 1) step = 1;
            if (tid % step == 0 && tid / step < residual) h++;       // bins 0, step, 2 step, ... get one more each
        }
        __syncthreads();
    }
    // inclusive scan over the 256 bins
    int x = h;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y2 = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y2; }
    if (lane == 31) s_part[wid] = x;
    __syncthreads();
    int pre = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) if (k < wid) pre += s_part[k];
    const int sum = pre + x;
    int v = __float2int_rn(__fmul_rn((float)sum, lut_scale));
    v = v < 0 ? 0 : v > 255 ? 255 : v;
    luts[((int64_t)f * tiles_x * tiles_y + tile) * 256 + tid] = (uint8_t)v;
}

constexpr int kPreTW = 64, kPreTH = 16;
__global__ void __launch_bounds__(256) pre_clahe_blur_kernel(const uint8_t* __restrict__ gray, const uint8_t* __restrict__ luts, int H, int W,
                                                             int tiles_x, int tiles_y, float inv_tw, float inv_th,
                                                             const uint8_t* __restrict__ gamma, uint8_t* __restrict__ out) {
    __shared__ uint8_t s_c[(kPreTH + 2) * (kPreTW + 2)];
    __shared__ uint8_t s_gamma[256];
    const int f = blockIdx.z, x0 = blockIdx.x * kPreTW, y0 = blockIdx.y * kPreTH, tid = threadIdx.x;
    s_gamma[tid] = gamma[tid];
    const uint8_t* __restrict__ g = gray + (int64_t)f * H * W;
    const uint8_t* __restrict__ L = luts + (int64_t)f * tiles_x * tiles_y * 256;
    for (int i = tid; i < (kPreTH + 2) * (kPreTW + 2); i += 256) {
        const int yy = i / (kPreTW + 2), xx = i - yy * (kPreTW + 2);
        const int y = reflect101(min(y0 - 1 + yy, H), H), x = reflect101(min(x0 - 1 + xx, W), W);   // (min: keeps out-of-range halo of edge tiles cheap)
        const float tyf = __fsub_rn(__fmul_rn((float)y, inv_th), 0.5f), txf = __fsub_rn(__fmul_rn((float)x, inv_tw), 0.5f);
        int ty1 = (int)floorf(tyf), tx1 = (int)floorf(txf);
        const float ya = __fsub_rn(tyf, (float)ty1), xa = __fsub_rn(txf, (float)tx1);
        const float ya1 = __fsub_rn(1.0f, ya), xa1 = __fsub_rn(1.0f, xa);
        int ty2 = min(ty1 + 1, tiles_y - 1), tx2 = min(tx1 + 1, tiles_x - 1);
        ty1 = max(ty1, 0); tx1 = max(tx1, 0);
        const int v = __ldg(g + (int64_t)y * W + x);
        const float l11 = (float)__ldg(L + (ty1 * tiles_x + tx1) * 256 + v), l12 = (float)__ldg(L + (ty1 * tiles_x + tx2) * 256 + v);
        const float l21 = (float)__ldg(L + (ty2 * tiles_x + tx1) * 256 + v), l22 = (float)__ldg(L + (ty2 * tiles_x + tx2) * 256 + v);
        const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa)), bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
        int r = __float2int_rn(__fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya)));
        s_c[i] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
    }
    __syncthreads();
    for (int i = tid; i < kPreTH * kPreTW; i += 256) {
        const int yy = i / kPreTW, xx = i - yy * kPreTW, y = y0 + yy, x = x0 + xx;
        if (y >= H || x >= W) continue;
        const uint8_t* c = s_c + yy * (kPreTW + 2) + xx;     // top-left of the 3x3 neighbourhood
        const int s = c[0] + 2 * c[1] + c[2] + 2 * c[kPreTW + 2] + 4 * c[kPreTW + 3] + 2 * c[kPreTW + 4] +
                      c[2 * (kPreTW + 2)] + 2 * c[2 * (kPreTW + 2) + 1] + c[2 * (kPreTW + 2) + 2];
        out[(int64_t)f * H * W + (int64_t)y * W + x] = s_gamma[(s + 8) >> 4];
    }
}

// =====================================================================================================
// K7  cv2.HOGDescriptor((32,32),(16,16),(8,8),(8,8),9,signed).compute  (REC:487-494,519), SURVEY A.7.
// One warp per window.  Gradient votes are staged in shared memory; each (block, cell, bin) accumulator has a
// FIXED owner lane that walks the block's pixels in raster order -> no float atomics, bit-reproducible runs.
// =====================================================================================================
__device__ __forceinline__ float fast_atan_deg(float y, float x) {
    const float sc = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * sc, p3 = -0.3258083974640975f * sc;
    const float p5 = 0.1555786518463281f * sc, p7 = -0.04432655554792128f * sc;
    float ax = fabsf(x), ay = fabsf(y), a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, ax + (float)DBL_EPSILON); c2 = c * c;
        a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    } else {
        c = __fdiv_rn(ax, ay + (float)DBL_EPSILON); c2 = c * c;
        a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

// The block histogram weight of pixel (i, j) of a 16x16 block for cell (cx, cy) is gauss(i) gauss(j) * wx(i, cx) * wy(j, cy):
// SEPARABLE.  wsep[i][c] = gauss(i) * (bilinear weight of cell c at position i, 0 when the cell is out of reach), built on the
// host (HOGCache::init: sigma = 4, cells of 8 px, neighbours outside [0,2) dropped).
struct HogConst {
    float wsep[16][2];
};

// v2: two separable stages instead of a gather per accumulator.  (1) lane = column x walks the 32 rows: gradient, magnitude,
// polynomial atan, the two orientation votes; each vote goes straight into Rv[(by, cy)][bin][x] with the VERTICAL weight of its
// row (<= 4 (block row, cell row) combinations per row, warp-uniform) -- the gradient planes are never stored.  (2) each of
// the 324 accumulators (block, cell, bin) is a 12-tap HORIZONTAL sum over Rv.  Then L2-Hys per block with warp reductions.
// Summation order differs from OpenCV's raster walk: features agree to ~1e-6 relative (tolerance 1e-4).  No float atomics:
// every Rv element has a single owner lane, so runs are bit-reproducible.
constexpr int kHogWarps = 4;
constexpr int kHogRvPitch = 33;                      // 32 columns + 1: conflict-free rows for the horizontal pass
__global__ void __launch_bounds__(kHogWarps * 32) k7_hog_kernel(const uint8_t* __restrict__ gray, const int32_t* __restrict__ n_ptr,
                                                               int n_max, HogConst hc, float* __restrict__ desc) {
    __shared__ __align__(16) uint8_t s_img[kHogWarps][32 * 32];
    __shared__ float s_rv[kHogWarps][6 * 9 * kHogRvPitch];
    __shared__ float s_hist[kHogWarps][9 * 36];
    __shared__ float s_ws[16][2];
    if (threadIdx.x < 32) s_ws[threadIdx.x >> 1][threadIdx.x & 1] = hc.wsep[threadIdx.x >> 1][threadIdx.x & 1];
    __syncthreads();
    const int wl = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int nwarps = gridDim.x * kHogWarps;
    const float angleScale = (float)(9.0 / (2.0 * 3.14159265358979323846));
    const float deg2rad = (float)(3.14159265358979323846 / 180.0);
    float* rv = s_rv[wl];
    for (int w = blockIdx.x * kHogWarps + wl; w < n; w += nwarps) {
        // 1024 B = 64 x 16 B: two 128-bit loads per lane
        const uint4* img4 = reinterpret_cast<const uint4*>(gray + (int64_t)w * 1024);
        uint4* s4 = reinterpret_cast<uint4*>(s_img[wl]);
        s4[lane] = __ldg(img4 + lane);
        s4[lane + 32] = __ldg(img4 + lane + 32);
        for (int i = lane; i < 6 * 9 * kHogRvPitch; i += 32) rv[i] = 0.f;
        __syncwarp();
        const int x = lane;
        const int xp = x == 0 ? 1 : x - 1, xn = x == 31 ? 30 : x + 1;           // BORDER_REFLECT_101
#pragma unroll 4
        for (int y = 0; y < 32; y++) {
            const int yp = y == 0 ? 1 : y - 1, yn = y == 31 ? 30 : y + 1;
            const float dx = (float)s_img[wl][y * 32 + xn] - (float)s_img[wl][y * 32 + xp];
            const float dy = (float)s_img[wl][yn * 32 + x] - (float)s_img[wl][yp * 32 + x];
            const float mag = __fsqrt_rn(dx * dx + dy * dy);
            const float ang = fast_atan_deg(dy, dx) * deg2rad;
            float t = ang * angleScale - 0.5f;
            int hidx = (int)floorf(t);
            t -= (float)hidx;
            if (hidx < 0) hidx += 9; else if (hidx >= 9) hidx -= 9;
            int h1 = hidx + 1; if (h1 >= 9) h1 = 0;
            const float g0 = mag * (1.f - t), g1 = mag * t;
            // rows of blocks by = band-1 (j = y - 8 by >= 8) and by = band (j < 8), band = y >> 3
            const int band = y >> 3;
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const int by = band - 1 + k;
                if (by < 0 || by > 2) continue;              // warp-uniform
                const int j = y - 8 * by;
#pragma unroll
                for (int cy = 0; cy < 2; cy++) {
                    const float wv = s_ws[j][cy];
                    if (wv == 0.f) continue;                 // warp-uniform (cell row out of reach)
                    float* r = rv + (by * 2 + cy) * 9 * kHogRvPitch + x;
                    r[hidx * kHogRvPitch] += g0 * wv;
                    r[h1 * kHogRvPitch] += g1 * wv;
                }
            }
        }
        __syncwarp();
        // 324 accumulators: descriptor index a = (bx*3 + by)*36 + (cx*2 + cy)*9 + bin  (blocks and cells column-major)
        for (int a = lane; a < 324; a += 32) {
            const int blk = a / 36, rr = a - blk * 36, cell = rr / 9, bin = rr - cell * 9;
            const int bx = blk / 3, by = blk - bx * 3, cx = cell >> 1, cy = cell & 1;
            const float* r = rv + ((by * 2 + cy) * 9 + bin) * kHogRvPitch + 8 * bx;
            float acc = 0.f;
            const int i0 = cx ? 4 : 0;                       // cell column 0 reaches i < 12, column 1 reaches i >= 4
#pragma unroll
            for (int i = 0; i < 12; i++) acc += r[i0 + i] * s_ws[i0 + i][cx];
            s_hist[wl][a] = acc;
        }
        __syncwarp();
        // L2-Hys per block (36 values): warp reductions
        float* o = desc + (int64_t)w * 324;
        for (int blk = 0; blk < 9; blk++) {
            const float* h = s_hist[wl] + blk * 36;
            float v0 = h[lane], v1 = lane < 4 ? h[32 + lane] : 0.f;
            float sum = v0 * v0 + v1 * v1;
#pragma unroll
            for (int of = 16; of > 0; of >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, of);
            float sc = 1.f / (__fsqrt_rn(sum) + 36 * 0.1f);
            v0 = fminf(v0 * sc, 0.2f); v1 = fminf(v1 * sc, 0.2f);
            sum = v0 * v0 + v1 * v1;
#pragma unroll
            for (int of = 16; of > 0; of >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, of);
            sc = 1.f / (__fsqrt_rn(sum) + 1e-3f);
            o[blk * 36 + lane] = v0 * sc;
            if (lane < 4) o[blk * 36 + 32 + lane] = v1 * sc;
        }
        __syncwarp();
    }
}

// =====================================================================================================
// K8  predictProbabilityLDAClassifiers + extractBestPredictions  (REC:565-577,627-641,342-347), SURVEY A.8.
// z = x . w_c + b_c in f64 (sklearn up-casts the f32 descriptors); one warp per window, W staged in shared memory.
// Decision on p = expit(z) (keeps the saturation tie rule).
// =====================================================================================================
__device__ __forceinline__ int lda_decide(const double z[6], double tol) {
    double best[6]; int tag[6];
#pragma unroll
    for (int c = 0; c < 6; c++) {
        double p1 = 1.0 / (1.0 + exp(-z[c])), p0 = 1.0 - p1;
        best[c] = p0 > p1 ? p0 : p1;
        tag[c] = p0 > p1 ? 0 : c + 1;
    }
    bool nosign = true;
#pragma unroll
    for (int c = 0; c < 6; c++) if (tag[c] != 0 && best[c] > tol) nosign = false;
    if (nosign) return 0;
    int lab = 0; double bv = 0; bool first = true;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        double key = tag[c] != 0 ? best[c] : -INFINITY;
        if (first || key > bv) { bv = key; lab = tag[c]; first = false; }
    }
    return lab;
}

__global__ void __launch_bounds__(256) k8_lda_kernel(const float* __restrict__ X, const int32_t* __restrict__ n_ptr, int n_max,
                                                     int nfeat, const double* __restrict__ W, const double* __restrict__ b,
                                                     double tol, double* __restrict__ logits, int32_t* __restrict__ labels) {
    extern __shared__ double s_W[];                         // [nfeat][6]
    for (int i = threadIdx.x; i < nfeat * 6; i += blockDim.x) s_W[i] = W[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += nwarps) {
        const float* x = X + (int64_t)w * nfeat;
        double z[6] = {0, 0, 0, 0, 0, 0};
        for (int f = lane; f < nfeat; f += 32) {
            double xv = (double)x[f];
#pragma unroll
            for (int c = 0; c < 6; c++) z[c] += xv * s_W[f * 6 + c];
        }
#pragma unroll
        for (int c = 0; c < 6; c++) z[c] = warp_sum(z[c]) + b[c];
        if (lane == 0) {
            if (logits) for (int c = 0; c < 6; c++) logits[(int64_t)w * 6 + c] = z[c];
            labels[w] = lda_decide(z, tol);
        }
    }
}

// K8 on the tensor cores -- the EVALUATION north_star asks for, not the product path.  z = X W + b with mma.sync.m16n8k8 TF32
// (the contraction is [n,324] x [324,6]: N = 6 pads to 8, far below a tcgen05 tile, so the warp-level MMA is the right tensor
// instruction here).  SPLIT = 1: plain TF32 (10-bit mantissas).  SPLIT = 3: x = xh + xl, w = wh + wl in TF32, z = xh wh + xh wl +
// xl wh with FP32 accumulation (the usual 3xTF32 emulation of FP32).  One warp per 16 windows; W (hi and lo parts, [328][8],
// zero padded) in shared memory.  Measured against the f64 FMA kernel in DESIGN.md (label flips, logit error, time).
__device__ __forceinline__ uint32_t to_tf32(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
__device__ __forceinline__ void mma_tf32(float c[4], const uint32_t a[4], const uint32_t b[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

template <int SPLIT>
__global__ void __launch_bounds__(128) k8_lda_tf32_kernel(const float* __restrict__ X, int n, int nfeat, const double* __restrict__ W,
                                                          const double* __restrict__ b, double tol, float* __restrict__ logits, int32_t* __restrict__ labels) {
    extern __shared__ float s_w[];                           // [2][kpad][8]: hi parts, then lo parts
    const int kpad = (nfeat + 7) & ~7;
    for (int i = threadIdx.x; i < kpad * 8; i += blockDim.x) {
        const int f = i >> 3, cidx = i & 7;
        const double w = (f < nfeat && cidx < 6) ? W[f * 6 + cidx] : 0.0;
        const float wh = __uint_as_float(to_tf32((float)w));
        s_w[i] = wh;
        s_w[kpad * 8 + i] = __uint_as_float(to_tf32((float)(w - (double)wh)));
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int w0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 16; w0 < n; w0 += nwarps * 16) {
        const int r0 = min(w0 + g, n - 1), r1 = min(w0 + g + 8, n - 1);
        const float* x0 = X + (int64_t)r0 * nfeat;
        const float* x1 = X + (int64_t)r1 * nfeat;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k0 = 0; k0 < kpad; k0 += 8) {
            const int ka = k0 + t, kb = k0 + t + 4;
            const float v0 = ka < nfeat ? __ldg(x0 + ka) : 0.f, v1 = ka < nfeat ? __ldg(x1 + ka) : 0.f;
            const float v2 = kb < nfeat ? __ldg(x0 + kb) : 0.f, v3 = kb < nfeat ? __ldg(x1 + kb) : 0.f;
            uint32_t ah[4] = {to_tf32(v0), to_tf32(v1), to_tf32(v2), to_tf32(v3)};
            uint32_t bh[2] = {__float_as_uint(s_w[ka * 8 + g]), __float_as_uint(s_w[kb * 8 + g])};
            if (SPLIT == 3) {
                uint32_t al[4] = {to_tf32(v0 - __uint_as_float(ah[0])), to_tf32(v1 - __uint_as_float(ah[1])),
                                  to_tf32(v2 - __uint_as_float(ah[2])), to_tf32(v3 - __uint_as_float(ah[3]))};
                uint32_t bl[2] = {__float_as_uint(s_w[kpad * 8 + ka * 8 + g]), __float_as_uint(s_w[kpad * 8 + kb * 8 + g])};
                mma_tf32(acc, al, bh);                       // small terms first
                mma_tf32(acc, ah, bl);
            }
            mma_tf32(acc, ah, bh);
        }
        // C fragment: acc[0], acc[1] = row g, columns 2t, 2t+1 ; acc[2], acc[3] = row g + 8.  Gather the 6 logits of a row into one lane.
        float z0[6], z1[6];
#pragma unroll
        for (int cidx = 0; cidx < 6; cidx++) {
            const int src = (lane & ~3) | (cidx >> 1);
            const float e0 = __shfl_sync(0xffffffffu, acc[cidx & 1], src), e1 = __shfl_sync(0xffffffffu, acc[2 + (cidx & 1)], src);
            z0[cidx] = e0 + (float)b[cidx]; z1[cidx] = e1 + (float)b[cidx];
        }
        if (t == 0) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int row = w0 + g + 8 * h;
                if (row < n) {
                    double zd[6];
#pragma unroll
                    for (int cidx = 0; cidx < 6; cidx++) { const float z = h ? z1[cidx] : z0[cidx]; zd[cidx] = (double)z; if (logits) logits[(int64_t)row * 6 + cidx] = z; }
                    labels[row] = lda_decide(zd, tol);
                }
            }
        }
    }
}

// K8b  reducer.transform + KNeighborsClassifier(k).predict  (REC:592-596).  One warp per query: Z = (x - xbar) S in
// f64, then every lane keeps its k best of the training rows it visits; the warp merges by (distance, index).
constexpr int kKnnMaxK = 8;
constexpr int kKnnMaxLabels = 16;                   // training labels 0..15 (tsd_set_knn checks)
__global__ void __launch_bounds__(128) k8_knn_kernel(const float* __restrict__ X, int n, int nfeat, const double* __restrict__ xbar,
                                                     const double* __restrict__ S, const double* __restrict__ Zt,
                                                     const int32_t* __restrict__ yt, int ntrain, int k,
                                                     double* __restrict__ Zout, int32_t* __restrict__ labels) {
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= n) return;
    const float* x = X + (int64_t)w * nfeat;
    double z[6] = {0, 0, 0, 0, 0, 0};
    for (int f = lane; f < nfeat; f += 32) {
        double xc = (double)x[f] - xbar[f];
#pragma unroll
        for (int c = 0; c < 6; c++) z[c] += xc * S[f * 6 + c];
    }
#pragma unroll
    for (int c = 0; c < 6; c++) z[c] = warp_sum(z[c]);
    if (lane == 0 && Zout) for (int c = 0; c < 6; c++) Zout[(int64_t)w * 6 + c] = z[c];
    double bd[kKnnMaxK]; int bi[kKnnMaxK];
#pragma unroll
    for (int j = 0; j < kKnnMaxK; j++) { bd[j] = INFINITY; bi[j] = 0x7fffffff; }
    for (int t = lane; t < ntrain; t += 32) {
        double d = 0;
#pragma unroll
        for (int c = 0; c < 6; c++) { double e = z[c] - Zt[(int64_t)t * 6 + c]; d += e * e; }
        if (d < bd[k - 1]) {                                // per-lane indices increase, so ties keep the smaller index
            int pos = k - 1;
            while (pos > 0 && bd[pos - 1] > d) { bd[pos] = bd[pos - 1]; bi[pos] = bi[pos - 1]; pos--; }
            bd[pos] = d; bi[pos] = t;
        }
    }
    // k rounds of warp arg-min over the lanes' current heads
    int votes[kKnnMaxLabels];
#pragma unroll
    for (int j = 0; j < kKnnMaxLabels; j++) votes[j] = 0;
    int head = 0;
    for (int r = 0; r < k; r++) {
        double d = head < k ? bd[head] : INFINITY; int idx = head < k ? bi[head] : 0x7fffffff;
        double bdv = d; int bidx = idx;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double od = __shfl_xor_sync(0xffffffffu, bdv, o); int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
            if (od < bdv || (od == bdv && oi < bidx)) { bdv = od; bidx = oi; }
        }
        if (idx == bidx && d == bdv) head++;
        if (bidx != 0x7fffffff) { int y = yt[bidx]; if (y >= 0 && y < kKnnMaxLabels) votes[y]++; }
    }
    if (lane == 0) {
        int lab = 0, bv = -1;
        for (int y = 0; y < kKnnMaxLabels; y++) if (votes[y] > bv) { bv = votes[y]; lab = y; }   // ties -> smallest label
        labels[w] = lab;
    }
}

// =====================================================================================================
// detection records (one line of resultado.txt, DET:501-508)
// =====================================================================================================
struct DetRec { int32_t frame, x1, y1, x2, y2, id, hundredths, reserved; };

// per-frame count of emitted survivors (survivors are CSR by surv_offsets); one warp per frame
__global__ void det_count_kernel(const uint8_t* __restrict__ emit, const int32_t* __restrict__ surv_offsets, int nframes,
                                 int32_t* __restrict__ counts, int32_t* __restrict__ det_offsets, unsigned* __restrict__ ticket) {
    int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f < nframes) {
        int c = 0;
        for (int i = surv_offsets[f] + lane; i < surv_offsets[f + 1]; i += 32) c += emit[i] != 0;
        c = warp_sum_i(c);
        if (lane == 0) counts[f] = c;
    }
    scan_by_last_block(counts, nframes, det_offsets, ticket);      // the last CTA to finish: CSR offsets of the records
}

__global__ void det_write_kernel(const uint8_t* __restrict__ emit, const int32_t* __restrict__ id, const int32_t* __restrict__ hundredths,
                                 const int4* __restrict__ coords, const int32_t* __restrict__ slots,
                                 const int32_t* __restrict__ surv_offsets, const int32_t* __restrict__ det_offsets, int nframes,
                                 int det_cap, DetRec* __restrict__ out, const int32_t* __restrict__ nwin_ptr, const int32_t* __restrict__ nsurv_ptr,
                                 int32_t* __restrict__ summary) {
    int f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (f == 0 && lane == 0 && summary) {                   // {windows, survivors, detections, 0} of this chunk, fetched in one copy
        summary[0] = *nwin_ptr; summary[1] = *nsurv_ptr; summary[2] = det_offsets[nframes]; summary[3] = 0;
    }
    if (f >= nframes) return;
    int o = det_offsets[f];
    for (int base = surv_offsets[f]; base < surv_offsets[f + 1]; base += 32) {
        int i = base + lane;
        bool e = i < surv_offsets[f + 1] && emit[i] != 0;
        unsigned m = __ballot_sync(0xffffffffu, e);
        if (e) {
            int r = o + __popc(m & ((1u << lane) - 1));
            if (r < det_cap) {
                int4 c = coords[slots ? slots[i] : i];
                out[r] = DetRec{f, c.x, c.y, c.z, c.w, id[i], hundredths[i], 0};
            }
        }
        o += __popc(m);
    }
}

__global__ void label_emit_kernel(const int32_t* __restrict__ lab, const int32_t* __restrict__ n_ptr, int n_max, uint8_t* __restrict__ emit) {
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) emit[i] = lab[i] != 0 ? 1 : 0;
}

// =====================================================================================================
// N4  the evaluators' matching loops (reporting only).
// eval_match: checkIfDetectionByTypeOnFileIsCorrectIncorrectDuplicated (DET:425-450) for every detection at once -- best ground
// truth of the same frame and type bucket by sqrt(f(d_TL) f(d_BR)) (first strict maximum), "correct" when it exceeds tol.  A
// ground truth beyond the similarity table (similarity below sqrt(f(simtab_n - 1)), which the host requires to be below tol) can
// never be the match of a correct detection and is skipped.  eval_tally_*: the per (frame, type) counts of getCorrectsAndWrongByTypeOnFile (DET:401-422).
// =====================================================================================================
struct EvalBox { int32_t frame, x1, y1, x2, y2, type; };     // type = bucket 0..5 (DET:371-386: anything that is not 1..5 lands in the sixth)

__global__ void eval_match_kernel(const EvalBox* __restrict__ det, int ndet, const EvalBox* __restrict__ gt, const int32_t* __restrict__ gt_offsets,
                                  int nframes, const double* __restrict__ simtab, int simtab_n, double tol, int32_t* __restrict__ status,
                                  int32_t* __restrict__ match, uint8_t* __restrict__ gt_hit, int32_t* __restrict__ tally) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ndet) return;
    const EvalBox d = det[i];
    double best = -INFINITY;
    int bi = -1;
    if (d.frame >= 0 && d.frame < nframes) {
        for (int g = gt_offsets[d.frame]; g < gt_offsets[d.frame + 1]; g++) {
            const EvalBox r = gt[g];
            if (r.type != d.type) continue;
            const int64_t ax = (int64_t)d.x1 - r.x1, ay = (int64_t)d.y1 - r.y1, bx = (int64_t)d.x2 - r.x2, by = (int64_t)d.y2 - r.y2;
            const int64_t da = ax * ax + ay * ay, db = bx * bx + by * by;
            if (da >= simtab_n || db >= simtab_n) continue;
            const double sim = sqrt(simtab[da] * simtab[db]);
            if (sim > best) { best = sim; bi = g; }
        }
    }
    const bool ok = bi >= 0 && best > tol;
    status[i] = ok ? 1 : 0;
    match[i] = ok ? bi : -1;
    if (ok) gt_hit[bi] = 1;
    if (d.frame >= 0 && d.frame < nframes) atomicAdd(&tally[(d.frame * 6 + d.type) * 4 + (ok ? 0 : 1)], 1);
}

__global__ void eval_tally_gt_kernel(const EvalBox* __restrict__ gt, int ngt, const uint8_t* __restrict__ gt_hit, int32_t* __restrict__ tally) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngt) return;
    const EvalBox r = gt[g];
    atomicAdd(&tally[(r.frame * 6 + r.type) * 4 + 3], 1);                 // expected
    if (!gt_hit[g]) atomicAdd(&tally[(r.frame * 6 + r.type) * 4 + 2], 1); // not detected
}

// precision_recall_curve's loop (evaluar_resultados.py:224-262): one thread per image walks that image's detections in the global
// (score-descending) order; bboxes_overlap (:53-89) with the "ignore" rule, LAST maximum (>=), a ground truth is matched once.
struct EvalGt { int32_t left, top, right, bottom, cls; };
struct EvalDt { int32_t left, top, right, bottom, index; };     // index = position in the globally sorted detection list

__global__ void eval_iou_kernel(const EvalDt* __restrict__ det, const int32_t* __restrict__ det_offsets, const EvalGt* __restrict__ gt,
                                const int32_t* __restrict__ gt_offsets, int nimages, double ovr, uint8_t* __restrict__ gt_used,
                                uint8_t* __restrict__ tp, uint8_t* __restrict__ fp) {
    const int im = blockIdx.x * blockDim.x + threadIdx.x;
    if (im >= nimages) return;
    const int g0 = gt_offsets[im], g1 = gt_offsets[im + 1];
    for (int k = det_offsets[im]; k < det_offsets[im + 1]; k++) {
        const EvalDt d = det[k];
        double maxovr = 0.0;
        int gsel = g0;
        const int64_t darea = (int64_t)(d.right - d.left + 1) * (int64_t)(d.bottom - d.top + 1);
        for (int g = g0; g < g1; g++) {
            const EvalGt r = gt[g];
            double covr = 0.0;
            const int w = min(d.right, r.right) - max(d.left, r.left);
            if (w > 0) {
                const int h = min(d.bottom, r.bottom) - max(d.top, r.top);
                if (h > 0) {
                    const int64_t inter = (int64_t)w * h;
                    const int64_t uni = r.cls == -1 ? darea : darea + (int64_t)(r.right - r.left + 1) * (int64_t)(r.bottom - r.top + 1) - inter;
                    covr = (double)inter / (double)uni;
                }
            }
            if (covr >= maxovr) { maxovr = covr; gsel = g; }
        }
        uint8_t t = 0, f = 0;
        if (g1 > g0 && maxovr > ovr) {
            if (gt[gsel].cls != -1) {
                if (!gt_used[gsel]) { t = 1; gt_used[gsel] = 1; } else f = 1;
            }
        } else f = 1;
        tp[d.index] = t; fp[d.index] = f;
    }
}

__global__ void fill_u8_kernel(uint8_t* p, int64_t n, uint8_t v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

}  // namespace tsd
