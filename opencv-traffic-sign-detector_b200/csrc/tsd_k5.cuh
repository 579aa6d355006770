// tsd_k5.cuh -- K5: cleanDuplicatedDetections (DET:177-223) as three stages (histograms, pair classes, fold).
//
//  k5_hist_kernel  : one WARP per window -> sparse min-max-normalised H-S histogram (calculateHistAndNormalize,
//                    DET:575-586): entries (bin << 16 | count) sorted by bin, f64 moments, pixel hash, and the energies
//                    of 25 bin groups (Cauchy-Schwarz bound used by k5_pairs).
//  k5_gram_kernel  : the pair classes of a frame of up to 128 windows from the Gram matrix of its count histograms on the tensor
//                    cores (u8 IMMA, exact integers; see the kernel's header) -- the default producer of the bit rows below.
//  k5_pairs_kernel : the CUDA-core producer, for the frames k5_gram leaves over (todo list) or all frames with TSD_GRAM=0.
//                    ALL pairs (i < j) of a frame's windows -> two BIT rows per item j over the earlier items i:
//                    del[j] (CORREL > tol: the newer window replaces the older one) and mrg[j] (tol*0.8823 <= CORREL <= tol).
//                    cv2.compareHist(CORREL) (DET:200-202) is decided from the EXACT integer dot product of the bin
//                    counts, which bounds the f64 value to ~1e-7; only pairs within 1e-6 of a threshold take the exact f64
//                    path, so every class equals the one the exact evaluation gives.
//  k5_fold_warp    : the sequential fold itself, one WARP per frame.  The survivor list is a bit set in list (= index)
//                    order, one 32-bit word per lane (<= 1024 windows per frame); an item without merge costs a handful of
//                    instructions (AND the item's rows with the alive set).  A merge (rare) averages the pixels, rebuilds
//                    the item's histogram, re-classifies it against the survivors after the merge position and -- once the
//                    item is final -- against every later item (their bit rows described the un-merged histogram).
//                    Pass 2 (corner similarity, DET:209-213) runs in the same warp from coordinates in shared memory.
//                    Persistent warps pull frames longest-first (k5_order); the merged item is re-classified with the same
//                    Cauchy-Schwarz pruning and the same software-pipelined exact dots as k5_pairs.
// The exact dots are bound by the latency of the entry loads (L2): one pair per pipeline stage, two stages in flight in
// ping-pong registers, 128-bit loads (2 x 4 entries per lane cover 256 bins).
#pragma once
#include "tsd_kernels.cuh"

namespace tsd {

constexpr int kHistGroups = 25;                      // group = bin / 120 (two H rows)
// k5_gram walks the bins in chunks of kGramKC; the histogram kernel records where each chunk starts in a window's sorted entry
// list (u16 cb[1..kGramChunks], cb[kGramChunks] = nnz; two per word) in kGramCbWords extra rows of the energy block
constexpr int kGramKC = 512;                         // bins per chunk: a multiple of 32 (boundaries = prefix popcounts of bitmap words)
constexpr int kGramChunks = (kHistBins + kGramKC - 1) / kGramKC;
constexpr int kGramCbWords = (kGramChunks + 1) / 2;
constexpr int kEnergyRows = kHistGroups + kGramCbWords;   // rows of the [rows][windows] energy block
static_assert(kGramKC % 32 == 0 && kEnergyRows <= 32, "chunk boundaries");
constexpr int kClsUnsure = 3;
// The todo work lists of k5_gram / k5_gram_big / k5_pairs keep (frame << 8) | (I << 4) | J in an int32: the batch entry points
// (tsd_enqueue_frames and the chains behind it, tsd_dedup) refuse batches of kMaxBatchFrames frames or more.
constexpr int kMaxBatchFrames = 1 << 23;
constexpr int kGramBM = 128;                           // windows per frame k5_gram handles / rows per block of k5_gram_big
// Statistics: pairs whose integer-dot classification came within 2e-6 of a threshold and were decided by the exact f64 evaluation
// (tsd_stat_unsure_pairs; the tests use it to prove that path is exercised).  Rare, so the atomic costs nothing.
__device__ unsigned long long g_unsure_pairs = 0;

__device__ __forceinline__ int classify(double sim, double tol, double lo) {
    return sim > tol ? 1 : ((lo <= sim && sim <= tol) ? 2 : 0);
}

// cv2.compareHist(h1, h2, HISTCMP_CORREL) from the sparse dot product and the cached moments (symmetric in h1, h2)
__device__ __forceinline__ double correl_from(double s12, double s1x, double Ax, double s1y, double Ay) {
    const double scale = 1.0 / (double)kHistBins;
    double num = s12 - s1x * s1y * scale;
    double den2 = Ax * Ay;                                   // (s11 - s1*s1*scale) * (s22 - s2*s2*scale)
    return fabs(den2) > DBL_EPSILON ? num / sqrt(den2) : 1.0;
}

// Class from the EXACT integer dot product I = sum_b cnt_x[b]*cnt_y[b].  The f64 value the reference computes is
// s12 = sum fl32(cnt_x a_x) * fl32(cnt_y a_y) = a_x a_y I (1 + e), |e| <= 2^-23 + O(1e-16); the class is decided here
// when the approximation is further than 2e-6 (relative to sqrt(denom2)) from both thresholds, else kClsUnsure.
__device__ __forceinline__ int classify_from_int_s(int I, double xA, double xrA, double xs1, float xa, double yA, double yrA, double ys1, float ya,
                                                   double tol, double lo) {
    const double scale = 1.0 / (double)kHistBins;
    const double den2 = xA * yA;
    if (!(fabs(den2) > DBL_EPSILON)) return classify(1.0, tol, lo);
    if (!(den2 > 0.0) || !(xA > 0.0) || !(yA > 0.0)) return kClsUnsure;
    const double num = (double)xa * (double)ya * (double)I - xs1 * ys1 * scale;
    const double r = xrA * yrA;                              // sqrt(denom2) to ~1e-16
    const double m = 2e-6 * r + 1e-300;
    const double hi_t = tol * r, lo_t = lo * r;
    if (num > hi_t + m) return 1;
    if (num < lo_t - m) return 0;
    if (num > lo_t + m && num < hi_t - m) return 2;
    return kClsUnsure;
}
__device__ __forceinline__ int classify_from_int(int I, const WinMeta& x, const WinMeta& y, double tol, double lo) {
    return classify_from_int_s(I, x.A, x.rA, x.s1, x.a, y.A, y.rA, y.s1, y.a, tol, lo);
}

// Cauchy-Schwarz bound from the group energies: can the pair (x, y) reach the merge band at all?
// ub >= s12 (energies are inflated by 1e-5), so (ub - s1x s1y / N) / sqrt(Ax Ay) >= CORREL; below lo -> class 0.
__device__ __forceinline__ bool prunable(float ub, const WinMeta& x, double s1y, double Ay, double rAy, double lo) {
    const double den2 = x.A * Ay;
    if (!(den2 > DBL_EPSILON) || !(x.A > 0.0) || !(Ay > 0.0)) return false;
    const double num_ub = (double)ub * 1.00001 - x.s1 * s1y * (1.0 / (double)kHistBins);
    return num_ub < lo * (x.rA * rAy) * 0.99999 - 1e-300;
}

__device__ __forceinline__ WinMeta load_meta_cg(const WinMeta* p) {      // 3 x 128-bit loads (metas are rewritten inside the fold: no __ldg)
    WinMeta m;
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(&m);
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2];
    return m;
}

// =====================================================================================================================
// Histogram of one window by one warp.  Scratch (per warp, shared memory):
//   occ[w]    .x occupancy bits of bins 32w .. 32w+31, .y occupied bins before word w -> rank(bin) = perfect hash into cnt[]
//             (one 64-bit load gives both halves of the rank)
//   cnt[r]    count of the r-th occupied bin;  binof[r] that bin;  binbuf[p] bin of pixel p
// The occupancy is first marked as one BYTE per bin with plain stores (no atomics: lanes whose bins share a word do not queue on it)
// in the space of cnt and binof, dead until pass B, and each lane then packs its 96 bytes into its three bit words.
// A lane owns groups of four consecutive pixels, g = lane + 32 k.
// CAP = capacity in pixels (640 for D=25, 1024 for D=32).
// =====================================================================================================================
template <int CAP>
struct __align__(16) HistScratch {
    uint32_t gsum[32];           // sum of count^2 per bin group (exact integers -> deterministic energies)
    uint2 occ[96];
    uint32_t cnt[CAP];           // (k5_hist stages the window's pixels here during pass A; the bin marks follow it)
    uint16_t binof[CAP];
    uint16_t binbuf[CAP];
    __device__ __forceinline__ uint8_t* mark() { return reinterpret_cast<uint8_t*>(cnt); }     // [96 * 32] over cnt + binof
    static_assert(sizeof(uint32_t) * CAP + sizeof(uint16_t) * CAP >= 96 * 32, "the bin marks must fit into cnt + binof");
};
// The pixels of the last group past npx (npx % 4 != 0) are marked in this bin: bit 31 of occupancy word 95, above the 3000 bins.
// It is left out of the ranks, so those pixels count into cnt[nnz], past the entries.
constexpr int kPadBin = 96 * 32 - 1;
static_assert(kPadBin >= kHistBins, "pad bin");

// calcHist's hue bin floor(H * 50 / 180.0) for H in [0, 180) without a table: (H * 5) / 18 == (H * 18205) >> 16 (checked below for
// every H; tsd_create checks the same expression against the host-built Tables::hbin and fails loudly if they ever differ)
__host__ __device__ constexpr int hue_bin(int H) { return (H * 18205) >> 16; }
constexpr bool hue_bin_ok() {
    for (int H = 0; H < 180; H++) if (hue_bin(H) != (H * 5) / 18) return false;
    return true;
}
static_assert(hue_bin_ok(), "hue_bin");

struct HsvLut {                 // per CTA: OpenCV's two division tables (RGB2HSV_b)
    int32_t sdiv[256], hdiv[256];
    __device__ __forceinline__ int sd(int v, int) const { return sdiv[v]; }
    __device__ __forceinline__ int hd(int d, int) const { return hdiv[d]; }
};
__device__ __forceinline__ void load_hsv_lut(HsvLut& t, const Tables* __restrict__ tab) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { t.sdiv[i] = tab->sdiv[i]; t.hdiv[i] = tab->hdiv[i]; }
}
// H-S histogram bin of one BGR pixel (cv2.cvtColor BGR2HSV + calcHist([0,1], [50,60], [0,180,0,256]), DET:577-580)
template <class LUT>
__device__ __forceinline__ int hs_bin(int b, int g, int r, const LUT& lut, int lane) {
    const int v = max(b, max(g, r)), m = min(b, min(g, r));
    const int d = v - m;
    int h = (v == r) ? (g - b) : (v == g) ? (b - r + 2 * d) : (r - g + 4 * d);
    const int S = (d * lut.sd(v, lane) + (1 << 11)) >> 12;
    h = (h * lut.hd(d, lane) + (1 << 11)) >> 12;
    const int H = h < 0 ? h + 180 : h;
    return hue_bin(H) * kHistS + ((S * kHistS) >> 8);        // floor(S*60/256.0) exactly (60/256 is a dyadic rational)
}

// Pass A over group g (pixels 4g .. 4g+3), given as the three little-endian words that hold its 12 bytes: bins (pixels past npx ->
// kPadBin) stored with one 64-bit store, and the pixel hash.
template <int CAP, class LUT>
__device__ __forceinline__ void hist_group(uint32_t q0, uint32_t q1, uint32_t q2, int g, int npx, const LUT& lut, HistScratch<CAP>& sw,
                                           int lane, uint32_t& hsh) {
    const int p0 = 4 * g;
    const uint32_t col[4] = {q0 & 0xffffffu, __funnelshift_r(q0, q1, 24) & 0xffffffu, __funnelshift_r(q1, q2, 16) & 0xffffffu, q2 >> 8};
    uint32_t bins[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        int bin = hs_bin((int)(col[j] & 255u), (int)((col[j] >> 8) & 255u), (int)(col[j] >> 16), lut, lane);
        const uint32_t hv = pix_hash32(p0 + j, col[j]);
        if (j == 0 || p0 + j < npx) hsh += hv;               // (p0 < npx for every group a lane processes)
        else bin = kPadBin;
        bins[j] = (uint32_t)bin;
    }
    *reinterpret_cast<uint2*>(&sw.binbuf[p0]) = make_uint2(bins[0] | (bins[1] << 16), bins[2] | (bins[3] << 16));
}

// px: window pixels (global; may have been rewritten by this warp -> plain loads), e: entries out (global, es words,
// zero-padded to a multiple of 4), meta out, Eg: optional group energies (E_T + w, stride e_stride).
// Returns nnz.  All 32 lanes must call.  On return sw.cnt / sw.binof hold the entries (used to fill a dense copy).
template <int CAP, class LUT>
__device__ __forceinline__ int hist_build_warp(const uint8_t* px, int npx, const LUT& lut, HistScratch<CAP>& sw,
                                               uint32_t* __restrict__ e, WinMeta* meta, float* Eg, int64_t e_stride, bool gram_aux = false) {
    const int lane = threadIdx.x & 31;
    sw.gsum[lane] = 0;
    // pass A: bin of every pixel + pixel hash.  A 4-byte aligned window (internal layout) is read as three words per group
    // (conflict-free LDS.32 when staged), the packed public layout byte by byte.  Two groups per lane in flight.
    uint32_t hsh = 0;
    const int ngroups = (npx + 3) >> 2;
    if ((reinterpret_cast<uintptr_t>(px) & 3) == 0) {
        const uint32_t* pw = reinterpret_cast<const uint32_t*>(px);
#pragma unroll 2
        for (int g = lane; g < ngroups; g += 32) hist_group(pw[3 * g], pw[3 * g + 1], pw[3 * g + 2], g, npx, lut, sw, lane, hsh);
    } else {
#pragma unroll 2
        for (int g = lane; g < ngroups; g += 32) {
            uint32_t q[3] = {0, 0, 0};
#pragma unroll
            for (int i = 0; i < 12; i++) if (12 * g + i < 3 * npx) q[i >> 2] |= (uint32_t)px[12 * g + i] << (8 * (i & 3));
            hist_group(q[0], q[1], q[2], g, npx, lut, sw, lane, hsh);
        }
    }
    __syncwarp();                                            // (the pixels, staged in cnt by k5_hist, are dead from here)
    uint8_t* const mark = sw.mark();
#pragma unroll
    for (int i = lane; i < 96 * 32 / 16; i += 32) reinterpret_cast<uint4*>(mark)[i] = make_uint4(0, 0, 0, 0);
    __syncwarp();
#pragma unroll 2
    for (int g = lane; g < ngroups; g += 32) {
        const uint2 bb = *reinterpret_cast<const uint2*>(&sw.binbuf[4 * g]);
        mark[bb.x & 0xffffu] = 1; mark[bb.x >> 16] = 1; mark[bb.y & 0xffffu] = 1; mark[bb.y >> 16] = 1;
    }
    __syncwarp();
    // the lane's 96 marks (bins 96 lane .. 96 lane + 95) -> its three occupancy words: (x * 0x01020408) >> 24 gathers the four 0/1
    // bytes of x into bits 0..3 (every other partial product falls below bit 24 or past bit 31)
    uint32_t wd[3] = {0, 0, 0};
    {
        const uint4* m4 = reinterpret_cast<const uint4*>(mark) + 6 * lane;
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const uint4 q = m4[k];
            const uint32_t x[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int t = 0; t < 4; t++) wd[k >> 1] |= ((x[t] * 0x01020408u) >> 24) << (4 * (4 * (k & 1) + t));
        }
    }
    if (lane == 31) wd[2] &= 0x7fffffffu;                   // the pad bin is no rank
    // per-word exclusive prefix popcounts (lane owns words 3*lane .. 3*lane+2)
    const int c0 = __popc(wd[0]), c1 = __popc(wd[1]), c2 = __popc(wd[2]);
    int incl = c0 + c1 + c2;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    const int excl = incl - (c0 + c1 + c2);
    const int nnz = __shfl_sync(0xffffffffu, incl, 31);
    sw.occ[3 * lane] = make_uint2(wd[0], (uint32_t)excl);
    sw.occ[3 * lane + 1] = make_uint2(wd[1], (uint32_t)(excl + c0));
    sw.occ[3 * lane + 2] = make_uint2(wd[2], (uint32_t)(excl + c0 + c1));
    const int nnz4 = (nnz + 3) & ~3;
    {                                                        // zero cnt[0 .. nnz] (cnt[nnz] takes the pad pixels) in 16-byte stores
        const int nz4 = (nnz + ((npx & 3) ? 4 : 3)) >> 2;    // <= CAP / 4 (pad pixels: npx % 4 != 0 and nnz <= npx)
        uint4* c4 = reinterpret_cast<uint4*>(sw.cnt);
        for (int i = lane; i < nz4; i += 32) c4[i] = make_uint4(0, 0, 0, 0);
    }
    __syncwarp();
    // pass B: counts through the rank hash; binof[rank] = bin (all writers of a rank store the same value)
#pragma unroll 2
    for (int g = lane; g < ngroups; g += 32) {
        const uint2 bb = *reinterpret_cast<const uint2*>(&sw.binbuf[4 * g]);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int bin = (int)(((j < 2 ? bb.x : bb.y) >> (16 * (j & 1))) & 0xffffu);
            const uint2 o = sw.occ[bin >> 5];
            const int r = (int)o.y + __popc(o.x & ((1u << (bin & 31)) - 1));
            atomicAdd(&sw.cnt[r], 1u);
            sw.binof[r] = (uint16_t)bin;
        }
    }
    __syncwarp();
    unsigned mx = 0;
    for (int i = lane; i < nnz; i += 32) mx = max(mx, sw.cnt[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    // normalize: scale = 1/(max-min) in f64 (min == 0: npx < 3000 bins), a = (float)scale (cv2.normalize NORM_MINMAX -> convertTo)
    const double scale = ((double)mx - 0.0) > DBL_EPSILON ? 1.0 / ((double)mx - 0.0) : 0.0;
    const float a = (float)scale;
    // entries in rank (= bin) order, lane-strided; moments per lane in that order, then a fixed shuffle tree (deterministic)
    double s1 = 0, s11 = 0;
    for (int r = lane; r < nnz4; r += 32) {
        uint32_t v = 0;
        if (r < nnz) {
            const uint32_t c = sw.cnt[r], bin = sw.binof[r];
            v = (bin << 16) | c;
            const double h = (double)((float)c * a);
            s1 += h; s11 += h * h;
            if (Eg) atomicAdd(&sw.gsum[(bin * 2185u) >> 18], c * c);     // bin / 120, exact for bin < 3000 (checked exhaustively)
        }
        e[r] = v;
    }
    s1 = warp_sum(s1); s11 = warp_sum(s11);
    hsh = warp_sum_u(hsh);
    if (Eg) {
        // E_g = sqrt(sum h^2) over the group, h = fl32(count * a) <= count * a * (1 + 2^-23): a * sqrt(sum count^2), inflated by
        // 1e-5, is an upper bound of it (only ever used as a bound: Cauchy-Schwarz pruning in k5_pairs / the fold)
        __syncwarp();
        if (lane < kHistGroups) Eg[(int64_t)lane * e_stride] = a * sqrtf((float)sw.gsum[lane]) * 1.00001f;
        else if (gram_aux && lane < kEnergyRows) {           // entry index where chunk c starts = occupied bins before bitmap word c * kGramKC / 32
            const int c1 = 2 * (lane - kHistGroups) + 1, c2 = c1 + 1;
            const uint32_t p1 = c1 < kGramChunks ? sw.occ[c1 * (kGramKC / 32)].y : (uint32_t)nnz;
            const uint32_t p2 = c2 < kGramChunks ? sw.occ[c2 * (kGramKC / 32)].y : (uint32_t)nnz;
            reinterpret_cast<uint32_t*>(Eg)[(int64_t)lane * e_stride] = p1 | (p2 << 16);
        }
    }
    if (lane == 0) {
        const double A = s11 - s1 * s1 * (1.0 / (double)kHistBins);
        WinMeta m;
        m.s1 = s1; m.s11 = s11; m.A = A; m.rA = sqrt(A); m.a = a; m.nnz = nnz; m.hash = hsh; m.pad_ = 0;
        *meta = m;
    }
    __syncwarp();
    return nnz;
}

template <int CAP, int kHistWarps, class LUT>
struct HistKSmem {
    LUT lut;
    HistScratch<CAP> w[kHistWarps];
};
template <int CAP, int kHistWarps, int MINB, class LUT>
__global__ void __launch_bounds__(kHistWarps * 32, MINB) k5_hist_kernel(const uint8_t* __restrict__ windows, const int32_t* __restrict__ n_ptr,
                                                                  int n_max, int npx, int ws, int es, const Tables* __restrict__ tab,
                                                                  uint32_t* __restrict__ entries, WinMeta* __restrict__ meta,
                                                                  float* __restrict__ E_T, int64_t e_stride) {
    constexpr int NCH = (CAP * 3 / 16 + 31) / 32;            // 128-bit chunks per lane covering one window
    static_assert(sizeof(uint32_t) * CAP >= NCH * 32 * 16, "the pixel staging area must fit into HistScratch::cnt");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HistKSmem<CAP, kHistWarps, LUT>& S = *reinterpret_cast<HistKSmem<CAP, kHistWarps, LUT>*>(smem_raw);
    const LUT& lut = S.lut;
    load_hsv_lut(S.lut, tab);
    __syncthreads();
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    HistScratch<CAP>& sw = S.w[wid];
    const int n = n_ptr ? min(*n_ptr, n_max) : n_max;
    const int nwarps = gridDim.x * kHistWarps;
    const bool staged = (ws & 15) == 0 && ((uintptr_t)windows & 15) == 0 && ws <= NCH * 32 * 16;
    if (!staged) {                                           // packed public layout: pixels straight from global memory
        for (int w = blockIdx.x * kHistWarps + wid; w < n; w += nwarps)
            hist_build_warp<CAP>(windows + (int64_t)w * ws, npx, lut, sw, entries + (int64_t)w * es, meta + w,
                                 E_T ? E_T + w : nullptr, e_stride, E_T != nullptr);
        return;
    }
    // internal layout: the NEXT window travels into registers (128-bit loads, all in flight together) while the current
    // one is processed from shared memory -- the kernel was bound by the latency of its byte loads
    const int nch = ws >> 4;
    uint4 r[NCH];
    // pixels are staged in the warp's own count array: pass A (the only reader of the pixels) ends before the counts are zeroed,
    // and the next window waits in registers until then
    uint4* s_px_w = reinterpret_cast<uint4*>(sw.cnt);
    int w = blockIdx.x * kHistWarps + wid;
    if (w < n) {
        const uint4* g = reinterpret_cast<const uint4*>(windows + (int64_t)w * ws);
#pragma unroll
        for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) r[k] = __ldg(g + lane + 32 * k);
    }
    for (; w < n; w += nwarps) {
#pragma unroll
        for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) s_px_w[lane + 32 * k] = r[k];
        __syncwarp();
        if (w + nwarps < n) {
            const uint4* g = reinterpret_cast<const uint4*>(windows + (int64_t)(w + nwarps) * ws);
#pragma unroll
            for (int k = 0; k < NCH; k++) if (lane + 32 * k < nch) r[k] = __ldg(g + lane + 32 * k);
        }
        hist_build_warp<CAP>(reinterpret_cast<const uint8_t*>(s_px_w), npx, lut, sw, entries + (int64_t)w * es, meta + w,
                             E_T ? E_T + w : nullptr, e_stride, E_T != nullptr);
    }
}

// =====================================================================================================================
// k5_pairs: one warp per item j (its dense histogram, u16, in shared memory); 32 earlier items per step, one per lane,
// pruned by the energy bound; surviving pairs are evaluated warp-wide (coalesced entry loads), two pairs in flight.
// Output: M[(base + j)][0..RW) = delete bits over il, M[(base + j)][RW..2RW) = merge bits.
// =====================================================================================================================
constexpr int kPairWarps = 4;                          // 4-warp CTAs: finer tail granularity than 8 (-6 %), same L1 sharing of the streamed entries
constexpr int kDenseLen = kHistBins + 8;

__device__ __forceinline__ double exact_s12_warp(const uint16_t* dense, float a_d, const uint32_t* eo, int nnz_o, float a_o) {
    const int lane = threadIdx.x & 31;
    double s12 = 0;
    for (int e = lane; e < nnz_o; e += 32) {
        const uint32_t v = __ldcg(eo + e);
        const float hd = (float)dense[v >> 16] * a_d;
        const float ho = (float)(v & 0xffffu) * a_o;
        s12 += (double)hd * (double)ho;
    }
    return warp_sum(s12);
}

// Items jl0 .. jl0 + kPairWarps - 1 of frame f against the earlier items in [i_lo, i_hi) (i_lo a multiple of 32).
template <int G>
__device__ __forceinline__ void k5_pairs_tile(const uint32_t* __restrict__ entries, const WinMeta* __restrict__ meta,
                                              const float* __restrict__ E_T, int64_t e_stride, const int32_t* __restrict__ offsets, int es, int RW,
                                              double tol, double lo, uint32_t* __restrict__ M, int32_t* __restrict__ frame_cost, int f, int jl0,
                                              int i_lo, int i_hi) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int base = offsets[f], n = offsets[f + 1] - base;
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int jl = jl0 + wid;
    if (jl >= n || jl == 0 || n > RW * 32 || i_lo >= jl) return;          // warps are independent: no block barrier below
    uint16_t* dense = reinterpret_cast<uint16_t*>(smem_raw) + (size_t)wid * kDenseLen;
    for (int b = lane; b < kDenseLen / 2; b += 32) reinterpret_cast<uint32_t*>(dense)[b] = 0;
    __syncwarp();
    const WinMeta mj = meta[base + jl];
    {
        const uint32_t* ej = entries + (int64_t)(base + jl) * es;
        for (int e = lane; e < mj.nnz; e += 32) { const uint32_t v = __ldg(ej + e); dense[v >> 16] = (uint16_t)(v & 0xffffu); }
    }
    const float Ej = lane < kHistGroups ? __ldg(E_T + (int64_t)lane * e_stride + base + jl) : 0.f;
    __syncwarp();
    uint32_t* Mrow = M + (int64_t)(base + jl) * 2 * RW;
    const int i_end = min(jl, i_hi);
    for (int i0 = i_lo; i0 < i_end; i0 += 32) {
        const int il = i0 + lane;
        const bool valid = il < i_end;
        const int wi = base + (valid ? il : 0);
        // lane-parallel bound for 32 earlier windows at once
        float ub = 0.f;
#pragma unroll
        for (int g = 0; g < kHistGroups; g++) ub += __shfl_sync(0xffffffffu, Ej, g) * __ldg(E_T + (int64_t)g * e_stride + wi);
        const WinMeta mi = meta[wi];
        int c = 0;
        bool need = false;
        if (valid) {
            const double den2 = mj.A * mi.A;
            if (!(fabs(den2) > DBL_EPSILON)) c = classify(1.0, tol, lo);          // compareHist's degenerate branch
            else need = !prunable(ub, mj, mi.s1, mi.A, mi.rA, lo);
        }
        unsigned todo = __ballot_sync(0xffffffffu, need);
        int Ik = 0;
        if (G == 1) {
            // One pair per pipeline stage, two stages in flight (ping-pong registers, no copies): every lane loads 2 x 4
            // consecutive entries (128-bit) of the pair, i.e. one stage covers 256 entries -- most windows -- with both
            // loads issued a full stage before they are consumed.  The kernel is bound by the latency of these loads.
            const uint4* ent4 = reinterpret_cast<const uint4*>(entries) + (int64_t)(base + i0) * (es >> 2);
            const int es4 = es >> 2;
            int kA, nA, kB, nB;
            const uint4 *eA, *eB;
            uint4 a0, a1, b0, b1;
#define PAIR_FETCH(K, N, E, V0, V1)                                                                          \
            do {                                                                                             \
                K = todo ? __ffs(todo) - 1 : -1;                                                             \
                todo &= todo - 1;                                                                            \
                N = K >= 0 ? (__shfl_sync(0xffffffffu, mi.nnz, K & 31) + 3) >> 2 : 0;                        \
                E = ent4 + (int64_t)(K & 31) * es4;                                                          \
                V0 = lane < N ? __ldg(E + lane) : make_uint4(0, 0, 0, 0);                                    \
                V1 = lane + 32 < N ? __ldg(E + lane + 32) : make_uint4(0, 0, 0, 0);                          \
            } while (0)
#define PAIR_DOT(V) ((int)dense[(V).x >> 16] * (int)((V).x & 0xffffu) + (int)dense[(V).y >> 16] * (int)((V).y & 0xffffu) + \
                     (int)dense[(V).z >> 16] * (int)((V).z & 0xffffu) + (int)dense[(V).w >> 16] * (int)((V).w & 0xffffu))
#define PAIR_COMPUTE(K, N, E, V0, V1)                                                                        \
            do {                                                                                             \
                int acc = PAIR_DOT(V0) + PAIR_DOT(V1);                                                       \
                for (int e = lane + 64; e < N; e += 32) { const uint4 v = __ldg(E + e); acc += PAIR_DOT(v); } \
                acc = warp_sum_i(acc);                                                                       \
                if (lane == K) Ik = acc;                                                                     \
            } while (0)
            PAIR_FETCH(kA, nA, eA, a0, a1);
            while (kA >= 0) {
                PAIR_FETCH(kB, nB, eB, b0, b1);
                PAIR_COMPUTE(kA, nA, eA, a0, a1);
                if (kB < 0) break;
                PAIR_FETCH(kA, nA, eA, a0, a1);
                PAIR_COMPUTE(kB, nB, eB, b0, b1);
            }
#undef PAIR_FETCH
#undef PAIR_DOT
#undef PAIR_COMPUTE
        } else {
        // Groups of up to G pairs; every lane loads 4 consecutive entries (128-bit) of each pair, so one load instruction
        // covers 128 entries per pair.  The first loads of group g+1 are issued BEFORE group g is reduced (software
        // pipelining across groups): the kernel is bound by the latency of these loads, not by their bandwidth.
        int kc[G], nc[G], kn[G], nn[G];
        const uint4 *ec[G], *en[G];
        uint4 vc[G], vn[G];
        bool have = todo != 0;
#pragma unroll
        for (int u = 0; u < G; u++) {
            kc[u] = todo ? __ffs(todo) - 1 : -1;
            todo &= todo - 1;                               // (0 & anything stays 0)
            nc[u] = kc[u] >= 0 ? (__shfl_sync(0xffffffffu, mi.nnz, kc[u] & 31) + 3) >> 2 : 0;          // uint4 count (zero padded)
            ec[u] = reinterpret_cast<const uint4*>(entries + (int64_t)(base + i0 + (kc[u] & 31)) * es);
            vc[u] = lane < nc[u] ? __ldg(ec[u] + lane) : make_uint4(0, 0, 0, 0);
        }
        while (have) {
            const bool have_next = todo != 0;
#pragma unroll
            for (int u = 0; u < G; u++) {                    // next group: pop + first loads (harmless when the group is empty)
                kn[u] = todo ? __ffs(todo) - 1 : -1;
                todo &= todo - 1;
                nn[u] = kn[u] >= 0 ? (__shfl_sync(0xffffffffu, mi.nnz, kn[u] & 31) + 3) >> 2 : 0;
                en[u] = reinterpret_cast<const uint4*>(entries + (int64_t)(base + i0 + (kn[u] & 31)) * es);
                vn[u] = lane < nn[u] ? __ldg(en[u] + lane) : make_uint4(0, 0, 0, 0);
            }
            int acc[G];
#pragma unroll
            for (int u = 0; u < G; u++)
                acc[u] = (int)dense[vc[u].x >> 16] * (int)(vc[u].x & 0xffffu) + (int)dense[vc[u].y >> 16] * (int)(vc[u].y & 0xffffu) +
                         (int)dense[vc[u].z >> 16] * (int)(vc[u].z & 0xffffu) + (int)dense[vc[u].w >> 16] * (int)(vc[u].w & 0xffffu);
            int nmax = nc[0];
#pragma unroll
            for (int u = 1; u < G; u++) nmax = max(nmax, nc[u]);
            for (int e = lane + 32; e < nmax; e += 32) {     // windows with more than 128 occupied bins
                uint4 v[G];
#pragma unroll
                for (int u = 0; u < G; u++) v[u] = e < nc[u] ? __ldg(ec[u] + e) : make_uint4(0, 0, 0, 0);
#pragma unroll
                for (int u = 0; u < G; u++)
                    acc[u] += (int)dense[v[u].x >> 16] * (int)(v[u].x & 0xffffu) + (int)dense[v[u].y >> 16] * (int)(v[u].y & 0xffffu) +
                              (int)dense[v[u].z >> 16] * (int)(v[u].z & 0xffffu) + (int)dense[v[u].w >> 16] * (int)(v[u].w & 0xffffu);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int u = 0; u < G; u++) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], o);
            }
#pragma unroll
            for (int u = 0; u < G; u++) {
                if (lane == kc[u]) Ik = acc[u];
                kc[u] = kn[u]; nc[u] = nn[u]; ec[u] = en[u]; vc[u] = vn[u];
            }
            have = have_next;
        }
        }
        if (need) c = classify_from_int(Ik, mj, mi, tol, lo);
        unsigned unsure = __ballot_sync(0xffffffffu, need && c == kClsUnsure);
        if (unsure && lane == 0) atomicAdd(&g_unsure_pairs, (unsigned long long)__popc(unsure));
        while (unsure) {                                    // rare: within 2e-6 of a threshold -> exact f64 evaluation
            const int k = __ffs(unsure) - 1;
            unsure &= unsure - 1;
            const int nnz_k = __shfl_sync(0xffffffffu, mi.nnz, k);
            const float a_k = __shfl_sync(0xffffffffu, mi.a, k);
            const double s12 = exact_s12_warp(dense, mj.a, entries + (int64_t)(base + i0 + k) * es, nnz_k, a_k);
            if (lane == k) c = classify(correl_from(s12, mj.s1, mj.A, mi.s1, mi.A), tol, lo);
        }
        const unsigned bd = __ballot_sync(0xffffffffu, valid && c == 1), bm = __ballot_sync(0xffffffffu, valid && c == 2);
        if (lane == 0) {
            Mrow[i0 >> 5] = bd; Mrow[RW + (i0 >> 5)] = bm;
            if (bm && frame_cost) atomicAdd(frame_cost + f, __popc(bm));     // merge-band pairs: the fold's cost predictor
        }
    }
}

// CTA = (frame, tile of kPairWarps items j).  With `todo` (the frames k5_gram left over: more than kGramBM windows, or a count that
// does not fit a byte) a small grid walks that list; without it the grid covers every (frame, tile).
template <int G, int MINB>
__global__ void __launch_bounds__(kPairWarps * 32, MINB) k5_pairs_kernel(const uint32_t* __restrict__ entries, const WinMeta* __restrict__ meta,
                                                                   const float* __restrict__ E_T, int64_t e_stride,
                                                                   const int32_t* __restrict__ offsets, int nframes, int es, int RW,
                                                                   int tiles_per_frame, double tol, double lo, uint32_t* __restrict__ M,
                                                                   int32_t* __restrict__ frame_cost, const int32_t* __restrict__ todo) {
    // todo items: (frame << 8) | (I << 4) | J = items of the 128-row block I against those of block J; I = J = 15 = the whole frame
    const int nf = todo ? todo[0] : nframes;
    for (int64_t item = blockIdx.x; item < (int64_t)nf * tiles_per_frame; item += gridDim.x) {
        const int fi = (int)(item / tiles_per_frame), tile = (int)(item - (int64_t)fi * tiles_per_frame);
        int f = fi, jl0 = tile * kPairWarps, i_lo = 0, i_hi = 0x7fffffff;
        if (todo) {
            const int t = todo[1 + fi];
            f = t >> 8;
            const int I = (t >> 4) & 15, J = t & 15;
            if (I != 15) {
                if (tile >= kGramBM / kPairWarps) continue;  // (CTA-uniform) a block has 128 items
                jl0 += I * kGramBM; i_lo = J * kGramBM; i_hi = i_lo + kGramBM;
            }
        }
        k5_pairs_tile<G>(entries, meta, E_T, e_stride, offsets, es, RW, tol, lo, M, frame_cost, f, jl0, i_lo, i_hi);
        __syncwarp();
    }
}

// =====================================================================================================================
// k5_gram: the same two bit rows from the GRAM MATRIX of a frame's count histograms on the tensor cores.
// The integer dot products I[j][i] = sum_b cnt_j[b] cnt_i[b] of ALL pairs of a frame are one matrix product C C^T with
// C = [n windows][3000 bins] -- exact in u8 x u8 -> s32 (mma.sync m16n8k32) on the low bytes of the counts, which is what the tile
// holds; the rare counts above 255 (a window dominated by one flat colour) are corrected exactly from the sparse lists before the
// classification.  Frames with more than kGramBM windows or more than kGramMaxBig such rows are appended to the todo list of
// k5_pairs.  One CTA per frame.  Per chunk of kGramKC bins the sparse entries are
// scattered into a dense u8 tile in shared memory (row = window, K-major): the entries a chunk needs are known from the
// boundaries k5_hist recorded, and travel into a per-warp pool one chunk ahead (cp.async, in flight during the tensor-core phase
// of the previous chunk); four lanes per row scatter them (rows 96..127 of a large frame are second rows of the first 32 groups).
// Each warp owns one 32 x 32 block of the lower triangle (2 x 2 ldmatrix.x4 + 8 IMMA per 32 bins) and, when there are fewer
// blocks than warps, one slice of K; the integer partial sums meet in shared memory, where the lane-per-pair classification
// (classify_from_int, f64 fallback within 2e-6 of a threshold) reads them.
// =====================================================================================================================
constexpr int kGramTinyMax = 24;                       // frames of up to this many windows go straight to k5_pairs
constexpr int kGramWarps = 12;                         // 96 four-lane groups; 6 lower-triangle 32 x 32 blocks x 2 K slices for n <= 96
constexpr int kGramGroups = kGramWarps * 8;
constexpr int kGramPitch = kGramKC + 16;               // bytes per tile row: an odd number of 16-byte units -> conflict-free ldmatrix
constexpr int kGramPoolBig = 300, kGramPoolSmall = 150;   // 16-byte pieces (4 entries) per warp and chunk: warps 0..3 (up to 16 rows) / the others;
constexpr int kGramPoolTotal = 4 * kGramPoolBig + (kGramWarps - 4) * kGramPoolSmall;   // the rare overflow is read from global memory
constexpr int kGramMaxBig = 16;                        // more such rows in one frame (flat frames): the frame goes to k5_pairs
constexpr int kGramIPitch = kGramBM + 4;               // words per row of the integer result matrix (aliases the tile)
static_assert((kGramPitch / 16) % 2 == 1 && kGramBM * kGramIPitch * 4 <= kGramBM * kGramPitch, "gram tile layout");
static_assert(kGramBM == kGramGroups + 32 && kGramWarps >= 10, "rows 96..127 are the second rows of groups 0..31; 10 blocks for n = 128");

struct __align__(16) GramSmem {
    unsigned char tile[kGramBM * kGramPitch];
    uint4 pool[kGramPoolTotal];                             // per warp: the next chunk's entries of its rows
    double A[kGramBM], rA[kGramBM], s1[kGramBM];
    float a[kGramBM];
    int32_t nnz[kGramBM];
    uint16_t cb[kGramBM][kGramChunks + 2];                  // cb[r][c] = first entry of chunk c in row r's list (cb[r][kGramChunks] = nnz)
    int32_t nbig;                                           // rows with a count that does not fit a byte (the tile holds count & 255;
    int32_t bigrow[kGramMaxBig];                            //  their pairs are corrected exactly before the classification)
};

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void mma_u8_16832(int (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// exact f64 s12 of (j, i) from the two sparse lists: the same terms in the same order as exact_s12_warp (bins missing in j add +0.0)
__device__ __forceinline__ double exact_s12_sparse_warp(const uint32_t* ej, int nnz_j, float a_j, const uint32_t* ei, int nnz_i, float a_i) {
    const int lane = threadIdx.x & 31;
    double s12 = 0;
    for (int e = lane; e < nnz_i; e += 32) {
        const uint32_t v = __ldcg(ei + e);
        const uint32_t bin = v >> 16;
        int lo_ = 0, hi_ = nnz_j;
        while (lo_ < hi_) { const int mid = (lo_ + hi_) >> 1; if ((__ldcg(ej + mid) >> 16) < bin) lo_ = mid + 1; else hi_ = mid; }
        uint32_t cj = 0;
        if (lo_ < nnz_j) { const uint32_t u = __ldcg(ej + lo_); if ((u >> 16) == bin) cj = u & 0xffffu; }
        const float hd = (float)cj * a_j;
        const float ho = (float)(v & 0xffffu) * a_i;
        s12 += (double)hd * (double)ho;
    }
    return warp_sum(s12);
}

// Copy the entries chunk c needs of one row per four-lane group into the warp's pool (packed group after group behind `fill`,
// each from its 16-byte aligned-down start).  off / sp = the row's first piece / pieces staged.  All 32 lanes call.
__device__ __forceinline__ void gram_issue(const uint16_t* cbrow, bool act, const uint32_t* er, int c, uint4* pool, int cap, int& fill,
                                           int& off, int& sp) {
    const int lane = threadIdx.x & 31, sub = lane & 3;
    const int lo_ = act ? (int)cbrow[c] : 0, hi_ = act ? (int)cbrow[c + 1] : 0;
    const int a4 = lo_ & ~3;
    const int np = hi_ > lo_ ? (hi_ - a4 + 3) >> 2 : 0;
    int incl = np;                                           // scan over the warp's 8 groups (the four lanes of a group hold the same value)
    int t = __shfl_up_sync(0xffffffffu, incl, 4); if (lane >= 4) incl += t;
    t = __shfl_up_sync(0xffffffffu, incl, 8); if (lane >= 8) incl += t;
    t = __shfl_up_sync(0xffffffffu, incl, 16); if (lane >= 16) incl += t;
    off = fill + incl - np;
    sp = max(0, min(np, cap - off));
    for (int pc = sub; pc < sp; pc += 4) cp_async16(pool + off + pc, er + a4 + 4 * pc);
    fill += __shfl_sync(0xffffffffu, incl, 31);
}

// Scatter the row's entries of chunk `ch` into its tile row (counts as bytes); the staged ones from the pool, the rest from global memory.
__device__ __forceinline__ void gram_scatter(const uint16_t* cbrow, int ch, const uint4* pool, int off, int sp, const uint32_t* er,
                                             unsigned char* trow, int k0) {
    const int sub = threadIdx.x & 3;
    const int e_lo = cbrow[ch], e_hi = cbrow[ch + 1];
    const int a4 = e_lo & ~3, e_st = min(e_hi, a4 + 4 * sp);
    const uint32_t* pw = reinterpret_cast<const uint32_t*>(pool + off) - a4;
    int e = e_lo + sub;
#pragma unroll 4
    for (; e < e_st; e += 4) {
        const uint32_t v = pw[e];
        trow[(int)(v >> 16) - k0] = (unsigned char)v;
    }
    for (; e < e_hi; e += 4) {                               // (rare) the warp's pool was full
        const uint32_t v = __ldg(er + e);
        trow[(int)(v >> 16) - k0] = (unsigned char)v;
    }
}

__global__ void __launch_bounds__(kGramWarps * 32, 2) k5_gram_kernel(const uint32_t* __restrict__ entries, const WinMeta* __restrict__ meta,
                                                                    const float* __restrict__ E_T, int64_t e_stride,
                                                                    const int32_t* __restrict__ offsets, int nframes, int es, int RW,
                                                                    double tol, double lo, uint32_t* __restrict__ M,
                                                                    int32_t* __restrict__ frame_cost, int32_t* __restrict__ todo, int32_t* __restrict__ big,
                                                                    int prefetch_ahead) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GramSmem& S = *reinterpret_cast<GramSmem*>(smem_raw);
    const int f = blockIdx.x;
    if (f >= nframes) return;
    const int base = offsets[f], n = offsets[f + 1] - base;
    if (n < 2 || n > RW * 32) return;                       // (CTA-uniform) nothing to classify / the general fold's frame
    if (n <= kGramTinyMax) {                                // a handful of windows (real MSER frames: ~4): a warp per item in k5_pairs costs a few
        if (threadIdx.x == 0) todo[1 + atomicAdd(todo, 1)] = (f << 8) | 0xff;     // microseconds, this CTA's six chunk rounds ~40
        return;
    }
    if (n > kGramBM) {                                      // k5_gram_big's frame: its block pairs (I, J), J <= I, go to that kernel's work list
        const int nbk = (n + kGramBM - 1) / kGramBM, np = nbk * (nbk + 1) / 2;
        __shared__ int s_pos;
        if (threadIdx.x == 0) s_pos = atomicAdd(big, np);
        __syncthreads();
        for (int q = threadIdx.x; q < np; q += blockDim.x) {
            int I = 0, r = q;
            while (r > I) { r -= I + 1; I++; }
            big[1 + s_pos + q] = (f << 8) | (I << 4) | r;
        }
        return;
    }
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    // scatter role: group = tid / 4 owns row `group` and (frames of more than 96 windows, groups 0..31) row group + 96
    const int grp = tid >> 2, sub = tid & 3;
    const int row0 = grp, row1 = grp + kGramGroups;
    const bool act0 = row0 < n, act1 = grp < 32 && row1 < n;
    const bool two = n > kGramGroups;                        // (CTA-uniform)
    const uint32_t* er0 = entries + (int64_t)(base + (act0 ? row0 : 0)) * es;
    const uint32_t* er1 = entries + (int64_t)(base + (act1 ? row1 : 0)) * es;
    if (tid == 0) S.nbig = 0;
    __syncthreads();
    if ((act0 && sub == 0) || (act1 && sub == 1)) {
        const int r = sub == 0 ? row0 : row1;
        const WinMeta m = meta[base + r];
        S.A[r] = m.A; S.rA[r] = m.rA; S.s1[r] = m.s1; S.a[r] = m.a; S.nnz[r] = m.nnz;
        if (m.nnz > 0 && m.a < 1.0f / 255.5f) {              // a = (float)(1 / max count): max count >= 256
            const int q = atomicAdd(&S.nbig, 1);
            if (q < kGramMaxBig) S.bigrow[q] = r;
        }
        // the row's chunk boundaries (written by k5_hist): every load address of the scatter is known in advance
        uint16_t* cbr = S.cb[r];
        cbr[0] = 0;
#pragma unroll
        for (int k = 0; k < kGramCbWords; k++) {
            const uint32_t wv = __ldg(reinterpret_cast<const uint32_t*>(E_T) + (int64_t)(kHistGroups + k) * e_stride + base + r);
            cbr[2 * k + 1] = (uint16_t)(wv & 0xffffu);
            if (2 * k + 2 <= kGramChunks) cbr[2 * k + 2] = (uint16_t)(wv >> 16);
        }
    }
    __syncthreads();
    if (S.nbig > kGramMaxBig) {                              // (CTA-uniform) left to k5_pairs
        if (tid == 0) todo[1 + atomicAdd(todo, 1)] = (f << 8) | 0xff;
        return;
    }
    const uint16_t* const cb0 = S.cb[act0 ? row0 : 0];
    const uint16_t* const cb1 = S.cb[act1 ? row1 : 0];
    uint4* const pool = S.pool + (wid < 4 ? wid * kGramPoolBig : 4 * kGramPoolBig + (wid - 4) * kGramPoolSmall);
    const int pcap = wid < 4 ? kGramPoolBig : kGramPoolSmall;
    int off0 = 0, sp0 = 0, off1 = 0, sp1 = 0;
    {
        int fill = 0;
        gram_issue(cb0, act0, er0, 0, pool, pcap, fill, off0, sp0);
        if (two) gram_issue(cb1, act1, er1, 0, pool, pcap, fill, off1, sp1);
    }
    {                                                        // pull a later frame's entry rows into L2 (this frame's were pulled by an earlier CTA)
        const int fp = f + prefetch_ahead;                   // = CTAs resident at once (2 per SM)
        if (fp < nframes) {
            const int bp = offsets[fp], np = min(offsets[fp + 1] - bp, kGramBM);
            for (int i = tid; i < np * 12; i += kGramWarps * 32) {
                const int r = i / 12, l = i - r * 12;
                if (l * 32 < es) asm volatile("prefetch.global.L2 [%0];" ::"l"(entries + (int64_t)(bp + r) * es + l * 32));
            }
        }
    }
    const int nb = (n + 31) >> 5, npad = nb * 32, npairs = nb * (nb + 1) / 2;
    // MMA role: this warp's 32 x 32 block of the lower triangle, 0:(0,0) 1:(1,0) 2:(1,1) 3:(2,0) ..., and its share of the 32-bin
    // steps: with fewer blocks than warps several warps split K of one block
    const int kslices = kGramWarps / npairs, kslice = wid / npairs;
    int bi = -1, bj = 0;
    if (kslice < kslices) { bi = 0; int q = wid - kslice * npairs; while (q > bi) { q -= bi + 1; bi++; } bj = q; }
    int acc[2][4][4];
#pragma unroll
    for (int mi = 0; mi < 2; mi++)
#pragma unroll
        for (int ni = 0; ni < 4; ni++)
#pragma unroll
            for (int q = 0; q < 4; q++) acc[mi][ni][q] = 0;
    const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(S.tile);
    // ldmatrix row addresses (8 x 16-byte rows per matrix = 8 windows x 16 bins): A fragment = (rows 0-7 | 8-15) x (bins 0-15 | 16-31)
    // in the order a0..a3; B fragments (both n8 halves of 16 windows) = (n 0-7: bins 0-15, 16-31), (n 8-15: bins 0-15, 16-31):
    // B[k][n] = C[n][k], so the K-major rows are read untransposed
    const uint32_t a_addr = tile_s + (uint32_t)((max(bi, 0) * 32 + (lane & 7) + ((lane >> 3) & 1) * 8) * kGramPitch + (lane >> 4) * 16);
    const uint32_t b_addr = tile_s + (uint32_t)((bj * 32 + (lane & 7) + (lane >> 4) * 8) * kGramPitch + ((lane >> 3) & 1) * 16);
    unsigned char* const trow0 = S.tile + (size_t)row0 * kGramPitch;
    unsigned char* const trow1 = S.tile + (size_t)(grp < 32 ? row1 : 0) * kGramPitch;
#pragma unroll 1
    for (int ch = 0; ch < kGramChunks; ch++) {
        const int k0 = ch * kGramKC;
        {                                                    // the group wipes its rows (rows n .. npad stay zero)
            const uint4 z = make_uint4(0, 0, 0, 0);
            if (row0 < npad) {
                uint4* r4 = reinterpret_cast<uint4*>(trow0);
#pragma unroll 4
                for (int i = sub; i < kGramPitch / 16; i += 4) r4[i] = z;
            }
            if (grp < 32 && row1 < npad) {
                uint4* r4 = reinterpret_cast<uint4*>(trow1);
#pragma unroll 4
                for (int i = sub; i < kGramPitch / 16; i += 4) r4[i] = z;
            }
        }
        cp_async_wait_all();
        __syncwarp();
        if (act0) gram_scatter(cb0, ch, pool, off0, sp0, er0, trow0, k0);
        if (act1) gram_scatter(cb1, ch, pool, off1, sp1, er1, trow1, k0);
        __syncwarp();                                        // the pool is free again
        if (ch + 1 < kGramChunks) {
            int fill = 0;
            gram_issue(cb0, act0, er0, ch + 1, pool, pcap, fill, off0, sp0);
            if (two) gram_issue(cb1, act1, er1, ch + 1, pool, pcap, fill, off1, sp1);
        }
        __syncthreads();
        if (bi >= 0) {
#pragma unroll 2
            for (int kk = kslice * 32; kk < kGramKC; kk += kslices * 32) {
                uint32_t a[2][4], b[2][4];
                ldmatrix_x4(a[0], a_addr + kk);
                ldmatrix_x4(a[1], a_addr + 16 * kGramPitch + kk);
                ldmatrix_x4(b[0], b_addr + kk);
                ldmatrix_x4(b[1], b_addr + 16 * kGramPitch + kk);
#pragma unroll
                for (int mi = 0; mi < 2; mi++)
#pragma unroll
                    for (int nj = 0; nj < 2; nj++) {
                        mma_u8_16832(acc[mi][nj * 2], a[mi], b[nj][0], b[nj][1]);
                        mma_u8_16832(acc[mi][nj * 2 + 1], a[mi], b[nj][2], b[nj][3]);
                    }
            }
        }
        __syncthreads();                                     // the tile is wiped (or becomes the result matrix) next
    }
    int32_t* sI = reinterpret_cast<int32_t*>(S.tile);
    if (kslices > 1) {
        for (int i = tid; i < npad * kGramIPitch; i += kGramWarps * 32) sI[i] = 0;
        __syncthreads();
    }
    if (bi >= 0) {
        const int g = lane >> 2, t = lane & 3;
#pragma unroll
        for (int mi = 0; mi < 2; mi++)
#pragma unroll
            for (int ni = 0; ni < 4; ni++) {
                const int row = bi * 32 + mi * 16 + g, col = bj * 32 + ni * 8 + 2 * t;
                int* d0 = &sI[row * kGramIPitch + col];
                int* d1 = &sI[(row + 8) * kGramIPitch + col];
                if (kslices > 1) {
                    atomicAdd(d0, acc[mi][ni][0]); atomicAdd(d0 + 1, acc[mi][ni][1]);
                    atomicAdd(d1, acc[mi][ni][2]); atomicAdd(d1 + 1, acc[mi][ni][3]);
                } else {
                    d0[0] = acc[mi][ni][0]; d0[1] = acc[mi][ni][1];
                    d1[0] = acc[mi][ni][2]; d1[1] = acc[mi][ni][3];
                }
            }
    }
    __syncthreads();
    if (S.nbig > 0) {                                        // (CTA-uniform, rare) counts above 255: the tile held count & 255
        // I_true - I_tile of a pair = sum over the bins where either count exceeds 255 of (c_r c_i - (c_r & 255)(c_i & 255)); every
        // such entry (r, bin) is visited once and corrects its pairs with all other rows i (a pair big in the SAME bin on both sides
        // is left to the lower row's entry)
        for (int q = wid; q < S.nbig; q += kGramWarps) {
            const int r = S.bigrow[q];
            const uint32_t* erow = entries + (int64_t)(base + r) * es;
            const int nz = S.nnz[r];
            for (int e0 = 0; e0 < nz; e0 += 32) {
                const uint32_t v = e0 + lane < nz ? __ldg(erow + e0 + lane) : 0u;
                unsigned mb = __ballot_sync(0xffffffffu, (v & 0xffffu) > 255u);
                while (mb) {
                    const int k = __ffs(mb) - 1;
                    mb &= mb - 1;
                    const uint32_t vb = __shfl_sync(0xffffffffu, v, k);
                    const uint32_t bin = vb >> 16;
                    const int cr = (int)(vb & 0xffffu);
                    for (int i = lane; i < n; i += 32) {
                        if (i == r) continue;
                        const uint32_t* ei = entries + (int64_t)(base + i) * es;
                        int lo_ = 0, hi_ = S.nnz[i];
                        const int nzi = hi_;
                        while (lo_ < hi_) { const int mid = (lo_ + hi_) >> 1; if ((__ldg(ei + mid) >> 16) < bin) lo_ = mid + 1; else hi_ = mid; }
                        if (lo_ >= nzi) continue;
                        const uint32_t u = __ldg(ei + lo_);
                        if ((u >> 16) != bin) continue;
                        const int ci = (int)(u & 0xffffu);
                        if (ci > 255 && i < r) continue;
                        atomicAdd(&sI[max(r, i) * kGramIPitch + min(r, i)], cr * ci - (cr & 255) * (ci & 255));
                    }
                }
            }
        }
        __syncthreads();
    }
    for (int jl = 1 + wid; jl < n; jl += kGramWarps) {       // one warp per item j, one earlier item per lane
        const double Aj = S.A[jl], rAj = S.rA[jl], s1j = S.s1[jl];
        const float aj = S.a[jl];
        uint32_t* Mrow = M + (int64_t)(base + jl) * 2 * RW;
        for (int i0 = 0; i0 < jl; i0 += 32) {
            const int il = i0 + lane;
            const bool valid = il < jl;
            const int ii = valid ? il : 0;
            int c = 0;
            if (valid) c = classify_from_int_s(sI[jl * kGramIPitch + ii], Aj, rAj, s1j, aj, S.A[ii], S.rA[ii], S.s1[ii], S.a[ii], tol, lo);
            unsigned unsure = __ballot_sync(0xffffffffu, valid && c == kClsUnsure);
            if (unsure && lane == 0) atomicAdd(&g_unsure_pairs, (unsigned long long)__popc(unsure));
            while (unsure) {                                // rare: within 2e-6 of a threshold -> exact f64 evaluation
                const int k = __ffs(unsure) - 1;
                unsure &= unsure - 1;
                const int ik = i0 + k;
                const double s12 = exact_s12_sparse_warp(entries + (int64_t)(base + jl) * es, S.nnz[jl], aj,
                                                         entries + (int64_t)(base + ik) * es, S.nnz[ik], S.a[ik]);
                if (lane == k) c = classify(correl_from(s12, s1j, Aj, S.s1[ik], S.A[ik]), tol, lo);
            }
            const unsigned bd = __ballot_sync(0xffffffffu, valid && c == 1), bm = __ballot_sync(0xffffffffu, valid && c == 2);
            if (lane == 0) {
                Mrow[i0 >> 5] = bd; Mrow[RW + (i0 >> 5)] = bm;
                if (bm && frame_cost) atomicAdd(frame_cost + f, __popc(bm));
            }
        }
    }
}

// =====================================================================================================================
// k5_gram_big: frames of 129 .. 1024 windows.  The Gram matrix C C^T of such a frame does not fit one CTA's shared memory, so it is
// cut into 128-row blocks and ONE CTA computes one block pair (I, J), J <= I: the classes of the items of block I against the
// (earlier) items of block J -- 128 x 128 pairs, 16 warps, each one 32 x 32 block of u8 IMMA (m16n8k32) accumulators.  Per chunk of
// kGramKC bins the rows of both blocks are scattered from their sparse lists into two dense u8 tiles (A = block I, B = block J;
// the same tile when I == J); the entries of the NEXT chunk are loaded into registers before the tensor-core phase of the current
// one (every load address is known from the chunk boundaries k5_hist recorded), so the L2 latency hides under the MMAs.
// Rows holding a count above 255 (flat windows; the tiles hold count & 255) are corrected exactly from the sparse lists, like in
// k5_gram; a block pair with more than kBigMaxRows such rows is appended to the todo list of the CUDA-core kernel (k5_pairs).
// Todo items (shared with k5_gram): (frame << 8) | (I << 4) | J, I = J = 15 standing for "the whole frame".
// =====================================================================================================================
constexpr int kBigWarps = 16;
constexpr int kBigRowsPerWarp = 2 * kGramBM / kBigWarps;                 // 256 rows (two blocks) over 16 warps
constexpr int kBigMaxRows = 32;
__host__ __device__ inline int todo_item(int f, int I, int J) { return (f << 8) | (I << 4) | J; }

struct __align__(16) GramBigSmem {
    unsigned char tile[2][kGramBM * kGramPitch];            // [0] = block I rows, [1] = block J rows; later the int32 result [128][kGramIPitch]
    double A[2 * kGramBM], rA[2 * kGramBM], s1[2 * kGramBM];
    float a[2 * kGramBM];
    int32_t nnz[2 * kGramBM];
    uint16_t cb[2 * kGramBM][kGramChunks + 2];
    int32_t nbig;
    int32_t bigrow[kBigMaxRows];                            // local row index 0..255 (>= 128: block J)
    uint32_t extra[2 * kGramBM][32];                        // entries 32 .. 63 of a row's range in the NEXT chunk (cp.async, lane-private slots)
};
static_assert(kGramBM * kGramIPitch * 4 <= 2 * kGramBM * kGramPitch, "result matrix aliases the tiles");
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(sa), "l"(gsrc) : "memory");
}

__global__ void __launch_bounds__(kBigWarps * 32, 1) k5_gram_big_kernel(const uint32_t* __restrict__ entries, const WinMeta* __restrict__ meta,
                                                                       const float* __restrict__ E_T, int64_t e_stride,
                                                                       const int32_t* __restrict__ offsets, int nframes, int es, int RW,
                                                                       double tol, double lo, uint32_t* __restrict__ M,
                                                                       int32_t* __restrict__ frame_cost, int32_t* __restrict__ todo, const int32_t* __restrict__ big) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GramBigSmem& S = *reinterpret_cast<GramBigSmem*>(smem_raw);
    const int nitems = big[0];                               // written by k5_gram (the launch before this one)
    for (int it = blockIdx.x; it < nitems; it += gridDim.x) {
    __syncthreads();                                         // (the previous item is complete: shared memory is free)
    const int item = big[1 + it];
    const int f = item >> 8, I = (item >> 4) & 15, J = item & 15;
    const int base = offsets[f], n = offsets[f + 1] - base;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    const bool diag = I == J;
    const int rowsI = min(kGramBM, n - I * kGramBM), rowsJ = min(kGramBM, n - J * kGramBM);
    // local row r: 0..127 = item I*128 + r, 128..255 = item J*128 + (r - 128) (unused when I == J)
    auto item_of = [&](int r) { return r < kGramBM ? I * kGramBM + r : J * kGramBM + (r - kGramBM); };
    auto row_ok = [&](int r) { return r < kGramBM ? r < rowsI : (!diag && r - kGramBM < rowsJ); };
    if (tid == 0) S.nbig = 0;
    __syncthreads();
    if (tid < 2 * kGramBM && row_ok(tid)) {
        const int r = tid, w = base + item_of(r);
        const WinMeta m = meta[w];
        S.A[r] = m.A; S.rA[r] = m.rA; S.s1[r] = m.s1; S.a[r] = m.a; S.nnz[r] = m.nnz;
        if (m.nnz > 0 && m.a < 1.0f / 255.5f) {              // a = (float)(1 / max count): max count >= 256
            const int k = atomicAdd(&S.nbig, 1);
            if (k < kBigMaxRows) S.bigrow[k] = r;
        }
        uint16_t* cbr = S.cb[r];
        cbr[0] = 0;
#pragma unroll
        for (int k = 0; k < kGramCbWords; k++) {
            const uint32_t wv = __ldg(reinterpret_cast<const uint32_t*>(E_T) + (int64_t)(kHistGroups + k) * e_stride + w);
            cbr[2 * k + 1] = (uint16_t)(wv & 0xffffu);
            if (2 * k + 2 <= kGramChunks) cbr[2 * k + 2] = (uint16_t)(wv >> 16);
        }
    }
    __syncthreads();
    if (S.nbig > kBigMaxRows) {                              // (CTA-uniform) flat frames: this block pair goes to k5_pairs
        if (tid == 0) todo[1 + atomicAdd(todo, 1)] = todo_item(f, I, J);
        continue;
    }
    // scatter role: warp w owns local rows w, w + 16, ... (16 rows); lane = entry within the row's chunk range
    uint32_t pre[kBigRowsPerWarp];
    auto load_chunk = [&](int c) {
#pragma unroll
        for (int k = 0; k < kBigRowsPerWarp; k++) {
            const int r = wid + kBigWarps * k;
            pre[k] = 0xffffffffu;
            if (row_ok(r)) {
                const int e = (int)S.cb[r][c] + lane, hi = (int)S.cb[r][c + 1];
                const uint32_t* er = entries + (int64_t)(base + item_of(r)) * es;
                if (e < hi) pre[k] = __ldg(er + e);
                if (e + 32 < hi) cp_async4(&S.extra[r][lane], er + e + 32);     // a window has ~25-40 occupied bins per 512-bin chunk
            }
        }
    };
    // MMA role: warp (bi, bj) = 32 x 32 block of the 128 x 128 pair matrix: rows bi*32.. of tile A x rows bj*32.. of tile B
    const int bi = wid >> 2, bj = wid & 3;
    const bool mma_on = !diag || bj <= bi;                   // diagonal block pair: lower triangle only
    int acc[2][4][4];
#pragma unroll
    for (int mi = 0; mi < 2; mi++)
#pragma unroll
        for (int ni = 0; ni < 4; ni++)
#pragma unroll
            for (int k = 0; k < 4; k++) acc[mi][ni][k] = 0;
    const uint32_t tA = (uint32_t)__cvta_generic_to_shared(S.tile[0]);
    const uint32_t tB = diag ? tA : (uint32_t)__cvta_generic_to_shared(S.tile[1]);
    const uint32_t a_addr = tA + (uint32_t)((bi * 32 + (lane & 7) + ((lane >> 3) & 1) * 8) * kGramPitch + (lane >> 4) * 16);
    const uint32_t b_addr = tB + (uint32_t)((bj * 32 + (lane & 7) + (lane >> 4) * 8) * kGramPitch + ((lane >> 3) & 1) * 16);
    load_chunk(0);
#pragma unroll 1
    for (int ch = 0; ch < kGramChunks; ch++) {
        const int k0 = ch * kGramKC;
        {                                                    // wipe both tiles (rows beyond n stay zero)
            const uint4 z = make_uint4(0, 0, 0, 0);
            uint4* t4 = reinterpret_cast<uint4*>(S.tile[0]);
            const int n16 = (diag ? 1 : 2) * kGramBM * kGramPitch / 16;
            for (int i = tid; i < n16; i += kBigWarps * 32) t4[i] = z;
        }
        cp_async_wait_all();                                 // this lane's own extra slots (written by its cp.async of the previous iteration)
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kBigRowsPerWarp; k++) {
            const int r = wid + kBigWarps * k;
            const uint32_t v = pre[k];
            unsigned char* trow = S.tile[r >> 7] + (size_t)(r & (kGramBM - 1)) * kGramPitch;
            if (v != 0xffffffffu) {
                trow[(int)(v >> 16) - k0] = (unsigned char)v;
                const int e1 = (int)S.cb[r][ch] + 32 + lane, hi = (int)S.cb[r][ch + 1];
                if (e1 < hi) { const uint32_t u = S.extra[r][lane]; trow[(int)(u >> 16) - k0] = (unsigned char)u; }
                if (e1 + 32 < hi) {                          // (rare) more than 64 entries of this row in the chunk
                    const uint32_t* er = entries + (int64_t)(base + item_of(r)) * es;
                    for (int e = e1 + 32; e < hi; e += 32) { const uint32_t u = __ldg(er + e); trow[(int)(u >> 16) - k0] = (unsigned char)u; }
                }
            }
        }
        __syncwarp();                                        // the extra slots are free again
        if (ch + 1 < kGramChunks) load_chunk(ch + 1);        // in flight during the tensor-core phase below
        __syncthreads();
        if (mma_on) {
#pragma unroll 2
            for (int kk = 0; kk < kGramKC; kk += 32) {
                uint32_t a[2][4], b[2][4];
                ldmatrix_x4(a[0], a_addr + kk);
                ldmatrix_x4(a[1], a_addr + 16 * kGramPitch + kk);
                ldmatrix_x4(b[0], b_addr + kk);
                ldmatrix_x4(b[1], b_addr + 16 * kGramPitch + kk);
#pragma unroll
                for (int mi = 0; mi < 2; mi++)
#pragma unroll
                    for (int nj = 0; nj < 2; nj++) {
                        mma_u8_16832(acc[mi][nj * 2], a[mi], b[nj][0], b[nj][1]);
                        mma_u8_16832(acc[mi][nj * 2 + 1], a[mi], b[nj][2], b[nj][3]);
                    }
            }
        }
        __syncthreads();                                     // the tiles are wiped (or become the result matrix) next
    }
    int32_t* sI = reinterpret_cast<int32_t*>(S.tile[0]);     // [row of block I][row of block J]
    if (mma_on) {
        const int g = lane >> 2, t = lane & 3;
#pragma unroll
        for (int mi = 0; mi < 2; mi++)
#pragma unroll
            for (int ni = 0; ni < 4; ni++) {
                const int row = bi * 32 + mi * 16 + g, col = bj * 32 + ni * 8 + 2 * t;
                int* d0 = &sI[row * kGramIPitch + col];
                int* d1 = &sI[(row + 8) * kGramIPitch + col];
                d0[0] = acc[mi][ni][0]; d0[1] = acc[mi][ni][1];
                d1[0] = acc[mi][ni][2]; d1[1] = acc[mi][ni][3];
            }
    }
    __syncthreads();
    if (S.nbig > 0) {                                        // (CTA-uniform, rare) counts above 255: the tiles held count & 255
        // every entry (row r, bin) with a count above 255 corrects its pairs with all rows of the OTHER block (all other rows of the
        // same block when I == J); a pair big in the same bin on both sides is left to the entry of the lower item
        for (int k = wid; k < S.nbig; k += kBigWarps) {
            const int r = S.bigrow[k], ir = item_of(r);
            const bool rI = r < kGramBM;
            const uint32_t* erow = entries + (int64_t)(base + ir) * es;
            const int nz = S.nnz[r];
            const int o0 = (diag || !rI) ? 0 : kGramBM, on = (diag || !rI) ? rowsI : rowsJ;      // the other side's local rows o0 .. o0+on
            for (int e0 = 0; e0 < nz; e0 += 32) {
                const uint32_t v = e0 + lane < nz ? __ldg(erow + e0 + lane) : 0u;
                unsigned mb = __ballot_sync(0xffffffffu, (v & 0xffffu) > 255u);
                while (mb) {
                    const int kb = __ffs(mb) - 1;
                    mb &= mb - 1;
                    const uint32_t vb = __shfl_sync(0xffffffffu, v, kb);
                    const uint32_t bin = vb >> 16;
                    const int cr = (int)(vb & 0xffffu);
                    for (int x = lane; x < on; x += 32) {
                        const int ro = o0 + x, io = item_of(ro);
                        if (io == ir) continue;
                        const uint32_t* ei = entries + (int64_t)(base + io) * es;
                        int lo_ = 0, hi_ = S.nnz[ro];
                        const int nzi = hi_;
                        while (lo_ < hi_) { const int mid = (lo_ + hi_) >> 1; if ((__ldg(ei + mid) >> 16) < bin) lo_ = mid + 1; else hi_ = mid; }
                        if (lo_ >= nzi) continue;
                        const uint32_t u = __ldg(ei + lo_);
                        if ((u >> 16) != bin) continue;
                        const int ci = (int)(u & 0xffffu);
                        if (ci > 255 && io < ir) continue;
                        // result cell: [local row in I][local row in J]; for I == J the lower triangle [later][earlier]
                        int cI, cJ;
                        if (diag) { cI = max(r, ro); cJ = min(r, ro); }
                        else { cI = rI ? r : ro; cJ = (rI ? ro : r) - kGramBM; }
                        atomicAdd(&sI[cI * kGramIPitch + cJ], cr * ci - (cr & 255) * (ci & 255));
                    }
                }
            }
        }
        __syncthreads();
    }
    // classification: one warp per item j of block I, one earlier item of block J per lane
    for (int rj = wid; rj < rowsI; rj += kBigWarps) {
        const int jl = I * kGramBM + rj;
        const double Aj = S.A[rj], rAj = S.rA[rj], s1j = S.s1[rj];
        const float aj = S.a[rj];
        uint32_t* Mrow = M + (int64_t)(base + jl) * 2 * RW;
        for (int i0 = 0; i0 < rowsJ; i0 += 32) {
            const int ri = i0 + lane, il = J * kGramBM + ri;
            const bool valid = ri < rowsJ && il < jl;
            if (J * kGramBM + i0 >= jl) break;               // (warp-uniform) nothing earlier than j in this word
            const int rs = diag ? (valid ? ri : 0) : kGramBM + (valid ? ri : 0);      // the earlier item's local row (metadata index)
            int c = 0;
            if (valid) c = classify_from_int_s(sI[rj * kGramIPitch + ri], Aj, rAj, s1j, aj, S.A[rs], S.rA[rs], S.s1[rs], S.a[rs], tol, lo);
            unsigned unsure = __ballot_sync(0xffffffffu, valid && c == kClsUnsure);
            if (unsure && lane == 0) atomicAdd(&g_unsure_pairs, (unsigned long long)__popc(unsure));
            while (unsure) {                                // rare: within 2e-6 of a threshold -> exact f64 evaluation
                const int k = __ffs(unsure) - 1;
                unsure &= unsure - 1;
                const int rk = diag ? i0 + k : kGramBM + i0 + k, ik = J * kGramBM + i0 + k;
                const double s12 = exact_s12_sparse_warp(entries + (int64_t)(base + jl) * es, S.nnz[rj], aj,
                                                         entries + (int64_t)(base + ik) * es, S.nnz[rk], S.a[rk]);
                if (lane == k) c = classify(correl_from(s12, s1j, Aj, S.s1[rk], S.A[rk]), tol, lo);
            }
            const unsigned bd = __ballot_sync(0xffffffffu, valid && c == 1), bm = __ballot_sync(0xffffffffu, valid && c == 2);
            if (lane == 0) {
                const int word = (J * kGramBM + i0) >> 5;
                Mrow[word] = bd; Mrow[RW + word] = bm;
                if (bm && frame_cost) atomicAdd(frame_cost + f, __popc(bm));
            }
        }
    }
    }
}

// Longest-processing-time-first order of the frames for the fold: key = 32 * (merge-band pairs) + windows, counting sort,
// descending.  One CTA.  Also resets the fold's work counter.
__global__ void __launch_bounds__(1024) k5_order_kernel(const int32_t* __restrict__ frame_cost, const int32_t* __restrict__ offsets, int nframes,
                                                        int32_t* __restrict__ order, int32_t* __restrict__ counter) {
    constexpr int NB = 2048;
    __shared__ int32_t hist[NB];
    for (int i = threadIdx.x; i < NB; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int f = threadIdx.x; f < nframes; f += blockDim.x) {
        const int key = min(NB - 1, 32 * (frame_cost ? frame_cost[f] : 0) + (offsets[f + 1] - offsets[f]));
        atomicAdd(&hist[NB - 1 - key], 1);                   // bucket 0 = heaviest
    }
    __syncthreads();
    {                                                        // exclusive prefix over the 2048 buckets: two per thread + a block scan
        __shared__ int32_t wsum[32];
        const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
        const int c0 = hist[2 * tid], c1 = hist[2 * tid + 1];
        int x = c0 + c1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) wsum[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int v = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += y; }
            wsum[lane] = v;
        }
        __syncthreads();
        const int excl = (wid ? wsum[wid - 1] : 0) + x - (c0 + c1);
        hist[2 * tid] = excl; hist[2 * tid + 1] = excl + c0;
        if (tid == 0) { counter[0] = 0; counter[1] = 0; }   // work counters of k5_fold_warp / k5_fold_cta
    }
    __syncthreads();
    for (int f = threadIdx.x; f < nframes; f += blockDim.x) {
        const int key = min(NB - 1, 32 * (frame_cost ? frame_cost[f] : 0) + (offsets[f + 1] - offsets[f]));
        const int pos = atomicAdd(&hist[NB - 1 - key], 1);
        order[pos] = f;
    }
}

// =====================================================================================================================
// The fold: one warp per frame.
// =====================================================================================================================
constexpr int kFoldWarps = TSD_FOLD_WARPS;                          // default warps (= frames in flight) per CTA; the kernel reads blockDim

template <int RMAX, int CAP>
struct FoldPass1Smem {           // merge workspace of the histogram pass
    uint16_t dense[kDenseLen];   // dense counts of the item being merged
    float eg[32];                // its group energies (Cauchy-Schwarz pruning, as in k5_pairs)
    uint32_t rowd[32], rowm[32]; // class bits of the merged item against up to 1024 others (delete / merge), by word
    uint32_t cand_big[RMAX <= CAP ? 1 : RMAX];   // compacted list (item | nnz << 16) of the others that survive the pruning; when it
    HistScratch<CAP> hs;                         // fits it lives in hs.cnt instead (dead once the dense copy is filled)
    __device__ __forceinline__ uint32_t* cand() { return RMAX <= CAP ? hs.cnt : cand_big; }
};

template <int RMAX, int CAP>
struct FoldWarpSmem {
    uint32_t hash[RMAX];         // current pixel hash of every item (both passes: pop-by-pixel-equality pre-filter)
    union {                      // the two passes never overlap: the coordinate pass reuses the merge workspace for the coordinates
        FoldPass1Smem<RMAX, CAP> p1;
        int4 coords[RMAX];       // pass 2: current coords of every survivor candidate (merged coords also go to global)
    };
};

// cv2.addWeighted(a, .5, b, .5, 0) on 4 packed bytes: round-half-even of (a+b)/2 (DET:219)
__device__ __forceinline__ uint32_t avg_rne4(uint32_t a, uint32_t b) {
    const uint32_t fl = (a & b) + (((a ^ b) >> 1) & 0x7f7f7f7fu);    // floor((a+b)/2) per byte
    return fl + ((a ^ b) & fl & 0x01010101u);                         // halves round to even
}

// item[slot_i] = avg(item[slot_i], item[slot_k]) in place, whole padded window (pad bytes stay 0); returns the new pixel hash
template <bool HASH>
__device__ __forceinline__ uint32_t merge_pixels_warp(uint8_t* ipx, const uint8_t* kpx, int ws, int npx) {
    const int lane = threadIdx.x & 31;
    uint4* a4 = reinterpret_cast<uint4*>(ipx);
    const uint4* b4 = reinterpret_cast<const uint4*>(kpx);
    for (int i = lane; i < (ws >> 4); i += 32) {
        uint4 a = __ldcg(a4 + i);
        const uint4 b = __ldcg(b4 + i);
        a.x = avg_rne4(a.x, b.x); a.y = avg_rne4(a.y, b.y); a.z = avg_rne4(a.z, b.z); a.w = avg_rne4(a.w, b.w);
        a4[i] = a;
    }
    __syncwarp();
    if (!HASH) return 0;                                     // pass 1 gets the hash from the histogram rebuild
    uint32_t hsh = 0;
    for (int p = lane; p < npx; p += 32) hsh += pix_hash32(p, (uint32_t)(ipx[3 * p] | (ipx[3 * p + 1] << 8) | (ipx[3 * p + 2] << 16)));
    return warp_sum_u(hsh);
}

// Classes of the merged item (dense histogram in sm.p1.dense, meta mj, energies sm.p1.eg) against the items whose bits are set in
// cmask (lane w = items 32w..32w+31), words [w0, w1].  Three steps: (1) lane-parallel Cauchy-Schwarz pruning, 32 items at a
// time (class 0 without touching their histograms), survivors are compacted into sm.p1.cand; (2) lane-parallel exact
// classification of the compact list; (3) results as bit words in sm.p1.rowd / sm.p1.rowm.
template <int RMAX, int CAP>
__device__ __forceinline__ void fold_classify_against(FoldWarpSmem<RMAX, CAP>& sm, const FoldParams& P, const WinMeta& mj, int base, unsigned cmask,
                                                      int w0, int w1) {
    const int lane = threadIdx.x & 31;
    sm.p1.rowd[lane] = 0; sm.p1.rowm[lane] = 0;
    uint32_t* cand = sm.p1.cand();
    __syncwarp();
    int ncand = 0;
    for (int t = w0; t <= w1; t++) {
        const unsigned aw = __shfl_sync(0xffffffffu, cmask, t);
        if (!aw) continue;
        const bool mine = (aw >> lane) & 1u;
        const int q = base + 32 * t + lane;
        int c = 0, nnz_q = 0;
        bool need = false;
        if (mine) {
            float ub = 0.f;
#pragma unroll
            for (int g = 0; g < kHistGroups; g++) ub += sm.p1.eg[g] * P.E_T[(int64_t)g * P.e_stride + q];
            const WinMeta mq = load_meta_cg(P.meta + q);
            nnz_q = mq.nnz;
            const double den2 = mj.A * mq.A;
            if (!(fabs(den2) > DBL_EPSILON)) c = classify(1.0, P.hist_tol, P.hist_lo);      // compareHist's degenerate branch
            else need = !prunable(ub, mj, mq.s1, mq.A, mq.rA, P.hist_lo);
        }
        const unsigned nb = __ballot_sync(0xffffffffu, need);
        if (need) cand[ncand + __popc(nb & ((1u << lane) - 1))] = (uint32_t)(32 * t + lane) | ((uint32_t)nnz_q << 16);
        ncand += __popc(nb);
        const unsigned bd = __ballot_sync(0xffffffffu, c == 1), bm = __ballot_sync(0xffffffffu, c == 2);
        if (lane == 0) { sm.p1.rowd[t] = bd; sm.p1.rowm[t] = bm; }
    }
    __syncwarp();
    // step 2: exact integer dots of the compact list, warp-wide and software-pipelined exactly like k5_pairs (one candidate per
    // stage, two stages in flight, 128-bit entry loads): the fold is bound by the latency of these loads.  Plain loads: entries of
    // items merged earlier in this frame were rewritten by this warp.
    const uint16_t* dense = sm.p1.dense;
    const uint4* ent4 = reinterpret_cast<const uint4*>(P.entries) + (int64_t)base * (P.es >> 2);
    const int es4 = P.es >> 2;
    for (int r0 = 0; r0 < ncand; r0 += 32) {
        const int nr = min(32, ncand - r0);
        int Ik = 0;
        int cA = 0, cB = 0, nA = 0, nB = 0;
        const uint4 *eA = ent4, *eB = ent4;
        uint4 a0, a1, b0, b1;
#define FOLD_FETCH(CI, N, E, V0, V1)                                                                         \
        do {                                                                                                 \
            const uint32_t info = cand[r0 + (CI)];                                                           \
            N = (int)((info >> 16) + 3) >> 2;                                                                \
            E = ent4 + (int64_t)(info & 0xffffu) * es4;                                                      \
            V0 = lane < N ? E[lane] : make_uint4(0, 0, 0, 0);                                                \
            V1 = lane + 32 < N ? E[lane + 32] : make_uint4(0, 0, 0, 0);                                      \
        } while (0)
#define FOLD_DOT(V) ((int)dense[(V).x >> 16] * (int)((V).x & 0xffffu) + (int)dense[(V).y >> 16] * (int)((V).y & 0xffffu) + \
                     (int)dense[(V).z >> 16] * (int)((V).z & 0xffffu) + (int)dense[(V).w >> 16] * (int)((V).w & 0xffffu))
#define FOLD_COMPUTE(CI, N, E, V0, V1)                                                                       \
        do {                                                                                                 \
            int acc = FOLD_DOT(V0) + FOLD_DOT(V1);                                                           \
            for (int e = lane + 64; e < N; e += 32) { const uint4 v = E[e]; acc += FOLD_DOT(v); }            \
            acc = warp_sum_i(acc);                                                                           \
            if (lane == (CI)) Ik = acc;                                                                      \
        } while (0)
        FOLD_FETCH(cA, nA, eA, a0, a1);
        while (cA < nr) {
            cB = cA + 1;
            if (cB < nr) FOLD_FETCH(cB, nB, eB, b0, b1);
            FOLD_COMPUTE(cA, nA, eA, a0, a1);
            if (cB >= nr) break;
            cA = cB + 1;
            if (cA < nr) FOLD_FETCH(cA, nA, eA, a0, a1);
            FOLD_COMPUTE(cB, nB, eB, b0, b1);
        }
#undef FOLD_FETCH
#undef FOLD_DOT
#undef FOLD_COMPUTE
        if (lane < nr) {                                     // lane-parallel classification (exact f64 only within 2e-6 of a threshold)
            const int ql = (int)(cand[r0 + lane] & 0xffffu), q = base + ql;
            const WinMeta mq = load_meta_cg(P.meta + q);
            int c = classify_from_int(Ik, mj, mq, P.hist_tol, P.hist_lo);
            if (c == kClsUnsure) {
                atomicAdd(&g_unsure_pairs, 1ull);
                const uint32_t* eo = P.entries + (int64_t)q * P.es;
                double s12 = 0;
                for (int i = 0; i < mq.nnz; i++) {
                    const uint32_t v = eo[i];
                    s12 += (double)((float)dense[v >> 16] * mj.a) * (double)((float)(v & 0xffffu) * mq.a);
                }
                c = classify(correl_from(s12, mj.s1, mj.A, mq.s1, mq.A), P.hist_tol, P.hist_lo);
            }
            if (c == 1) atomicOr(&sm.p1.rowd[ql >> 5], 1u << (ql & 31));
            else if (c == 2) atomicOr(&sm.p1.rowm[ql >> 5], 1u << (ql & 31));
        }
        __syncwarp();
    }
    __syncwarp();
}

__device__ __forceinline__ bool pixels_equal_warp(const uint8_t* a, const uint8_t* b, int ws) {
    const int lane = threadIdx.x & 31;
    const uint4* a4 = reinterpret_cast<const uint4*>(a);
    const uint4* b4 = reinterpret_cast<const uint4*>(b);
    bool eq = true;
    for (int i = lane; i < (ws >> 4); i += 32) {
        const uint4 x = __ldcg(a4 + i), y = __ldcg(b4 + i);
        eq &= x.x == y.x && x.y == y.y && x.z == y.z && x.w == y.w;
    }
    return __all_sync(0xffffffffu, eq);
}

// calculateMeanMasks' running average (DET:44-52): per sign type, mask = first window, then mask = addWeighted(window, .5, mask, .5)
// for every further window IN ORDER (the result depends on the order: it is the caller's os.listdir order).  One warp per
// group; the bytes are independent, so each lane folds its own 16-byte chunks through the whole list.  Packed layout.
__global__ void __launch_bounds__(32) mean_windows_kernel(const uint8_t* __restrict__ windows, const int32_t* __restrict__ group_offsets,
                                                          int ngroups, int nbytes, uint8_t* __restrict__ mean_out) {
    const int g = blockIdx.x, lane = threadIdx.x;
    if (g >= ngroups) return;
    const int w0 = group_offsets[g], w1 = group_offsets[g + 1];
    for (int i = lane * 4; i < nbytes; i += 128) {           // 4 bytes per lane per step (packed windows are only 1-byte aligned)
        const int nb = min(4, nbytes - i);
        uint32_t m = 0;
        for (int w = w0; w < w1; w++) {
            const uint8_t* p = windows + (int64_t)w * nbytes + i;
            uint32_t v = 0;
            for (int k = 0; k < nb; k++) v |= (uint32_t)__ldg(p + k) << (8 * k);
            m = (w == w0) ? v : avg_rne4(v, m);
        }
        for (int k = 0; k < nb; k++) mean_out[(int64_t)g * nbytes + i + k] = (uint8_t)(m >> (8 * k));
    }
}

// pop-by-pixel-equality (DET:183-185,471-477) on the alive bit set A (lane w = items 32w..32w+31, list order = index order):
// for every marked position p, in increasing order, remove the FIRST alive entry whose pixels equal p's.  Returns new A.
template <int RMAX, int CAP>
__device__ __forceinline__ unsigned fold_apply_deletions(unsigned A, unsigned D, const FoldWarpSmem<RMAX, CAP>& sm, const uint8_t* windows,
                                                         int base, int ws) {
    const int lane = threadIdx.x & 31;
    unsigned lanes = __ballot_sync(0xffffffffu, D != 0);
    while (lanes) {
        const int L = __ffs(lanes) - 1;
        lanes &= lanes - 1;
        unsigned w = __shfl_sync(0xffffffffu, D, L);
        while (w) {
            const int bit = __ffs(w) - 1;
            w &= w - 1;
            const int p = 32 * L + bit;
            const uint32_t hp = sm.hash[p];
            int victim = p;
            for (int t = 0; t <= L && victim == p; t++) {
                unsigned aw = __shfl_sync(0xffffffffu, A, t);
                if (t == L) aw &= (1u << bit) - 1;
                const int q = 32 * t + lane;
                unsigned cm = __ballot_sync(0xffffffffu, ((aw >> lane) & 1u) && sm.hash[q] == hp);
                while (cm) {                                // candidates in list order; hash collisions are verified away
                    const int qq = 32 * t + __ffs(cm) - 1;
                    cm &= cm - 1;
                    if (pixels_equal_warp(windows + (int64_t)(base + qq) * ws, windows + (int64_t)(base + p) * ws, ws)) { victim = qq; break; }
                }
            }
            if (lane == (victim >> 5)) A &= ~(1u << (victim & 31));
        }
    }
    return A;
}


// Pass 2 of the fold (corner similarity, DET:209-213) of one frame by one warp: A1 = survivors of pass 1 (bit set, lane w = items
// 32w .. 32w+31, list order = item order).  Coordinates live in shared memory (overlaying the pass-1 workspace).  Returns the survivors.
template <int RMAX, int CAP>
__device__ __forceinline__ unsigned fold_coord_pass(unsigned A1, FoldWarpSmem<RMAX, CAP>& sm, const FoldParams& P, int base, int n, int sim_cut) {
    const int lane = threadIdx.x & 31;
    const int nwords = (n + 31) >> 5;
    const int ws = P.ws;
    __syncwarp();
    for (int p = lane; p < n; p += 32) sm.coords[p] = P.coords[base + p];      // overlays the pass-1 workspace
    __syncwarp();
    unsigned A2 = 0;
    const double tol = P.coord_tol, lo = P.coord_lo;
    for (int tj = 0; tj < nwords; tj++) {
        unsigned wj = __shfl_sync(0xffffffffu, A1, tj);
        while (wj) {
            const int j = 32 * tj + __ffs(wj) - 1;
            wj &= wj - 1;
            int4 ic = sm.coords[j];
            unsigned D = 0;
            bool dirty = false;
            int start = 0;                           // first list position still to scan
            int t = 0;
            while (t <= tj) {
                unsigned aw = __shfl_sync(0xffffffffu, A2, t);
                if (t == (start >> 5)) aw &= ~((1u << (start & 31)) - 1);
                if (!aw) { t++; continue; }
                int c = 0;
                if ((aw >> lane) & 1u) c = classify(coord_sim(ic, sm.coords[32 * t + lane], P.simtab, sim_cut), tol, lo);
                const unsigned bd = __ballot_sync(0xffffffffu, c == 1), bmm = __ballot_sync(0xffffffffu, c == 2);
                if (!bmm) { if (lane == t) D |= bd; t++; continue; }
                // ---- merge (DET:217-221): pixels, coords; later comparisons use the updated item ----
                const int bit = __ffs(bmm) - 1, fm = 32 * t + bit;
                if (lane == t) D |= (bd & ((1u << bit) - 1)) | (1u << bit);
                const uint32_t hsh = merge_pixels_warp<true>(P.windows + (int64_t)(base + j) * ws, P.windows + (int64_t)(base + fm) * ws, ws, P.npx);
                const int4 kc = sm.coords[fm];
                ic = make_int4((ic.x + kc.x) >> 1, (ic.y + kc.y) >> 1, (ic.z + kc.z) >> 1, (ic.w + kc.w) >> 1);
                if (lane == 0) sm.hash[j] = hsh;
                dirty = true;
                start = fm + 1;
                t = start >> 5;
                __syncwarp();
            }
            if (dirty) {
                if (lane == 0) { sm.coords[j] = ic; P.coords[base + j] = ic; P.meta[base + j].hash = sm.hash[j]; }
                __syncwarp();
            }
            if (__any_sync(0xffffffffu, D != 0)) A2 = fold_apply_deletions<RMAX, CAP>(A2, D, sm, P.windows, base, ws);
            if (lane == (j >> 5)) A2 |= 1u << (j & 31);
        }
    }
    return A2;
}

// survivors -> list (slots in list order) + count of frame f.  One warp.
__device__ __forceinline__ void fold_emit_survivors(unsigned A, const FoldParams& P, int f, int base) {
    const int lane = threadIdx.x & 31;
    const int cnt = __popc(A);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    int o = incl - cnt;
    unsigned w = A;
    while (w) { const int bit = __ffs(w) - 1; w &= w - 1; P.list[base + o++] = base + 32 * lane + bit; }
    if (lane == 31) P.out_count[f] = incl;
    __syncwarp();
}

// Frames of more than n_skip windows (up to 1024) are k5_fold_cta's: it is launched beside this kernel on the same order list.
template <int RMAX, int CAP>
__global__ void __launch_bounds__(kFoldWarps * 32, TSD_FOLD_MINB) k5_fold_warp_kernel(FoldParams P, int nframes, uint32_t* M, int RW, int sim_cut,
                                                                       const int32_t* __restrict__ order, int32_t* counter, int n_skip) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    HsvLut& lut = *reinterpret_cast<HsvLut*>(smem_raw);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    FoldWarpSmem<RMAX, CAP>& sm = reinterpret_cast<FoldWarpSmem<RMAX, CAP>*>(smem_raw + ((sizeof(HsvLut) + 15) & ~15))[wid];
    load_hsv_lut(lut, P.tab);
    for (int b = lane; b < kDenseLen / 2; b += 32) reinterpret_cast<uint32_t*>(sm.p1.dense)[b] = 0;
    __syncthreads();
    const int ws = P.ws, es = P.es;
    // persistent warps pull frames from a shared counter in longest-first order (k5_order_kernel): the heavy frames (many
    // merges) start first and the light ones fill in behind them
    while (true) {
        int idx = 0;
        if (lane == 0) idx = atomicAdd(counter, 1);
        idx = __shfl_sync(0xffffffffu, idx, 0);
        if (idx >= nframes) break;
        const int f = order[idx];
        const int base = P.offsets[f], n = P.offsets[f + 1] - base;
        if (n <= RW * 32 && n <= 1024 && n > n_skip) continue;     // k5_fold_cta's frame
        if (n > RMAX || n > RW * 32) { if (lane == 0) P.out_count[f] = -1; continue; }    // host picks RMAX / RW large enough
        for (int p = lane; p < n; p += 32) sm.hash[p] = P.meta[base + p].hash;
        bool dense_clean = false;                            // the previous frame's pass 2 overlaid the dense scratch: wiped at the first merge
        __syncwarp();
        const int nwords = (n + 31) >> 5;
        unsigned A = 0;                                      // survivors, list order = item order
        if (P.do_hist) {
            const uint32_t* Mf = M + (int64_t)base * 2 * RW;
            unsigned nd = 0, nm = 0;
            if (n > 1 && lane < RW) { nd = __ldcg(Mf + 2 * RW + lane); nm = __ldcg(Mf + 3 * RW + lane); }
            if (n > 0 && lane == 0) A = 1u;
            for (int j = 1; j < n; j++) {
                unsigned vd = nd, vm = nm;
                if (j + 1 < n && lane < RW) { nd = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + lane); nm = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + RW + lane); }
                unsigned D = 0, scan = 0xffffffffu;
                bool dirty = false;
                int4 ic = make_int4(0, 0, 0, 0);
                WinMeta mj;
                mj.nnz = 0;
                const int slot = base + j;
                while (true) {
                    const unsigned m = vm & A & scan, d = vd & A & scan;
                    const unsigned bm = __ballot_sync(0xffffffffu, m != 0);
                    if (!bm) { D |= d; break; }
                    // ---- merge with the first survivor (list order) in the merge band (DET:217-221) ----
                    const int L = __ffs(bm) - 1;
                    const int bit = __ffs(__shfl_sync(0xffffffffu, m, L)) - 1;
                    const int fm = 32 * L + bit;
                    if (lane < L) D |= d;
                    else if (lane == L) D |= (d & ((1u << bit) - 1)) | (1u << bit);
                    uint8_t* ipx = P.windows + (int64_t)slot * ws;
                    uint32_t* ient = P.entries + (int64_t)slot * es;
                    if (!dense_clean) {
                        for (int b = lane; b < kDenseLen / 2; b += 32) reinterpret_cast<uint32_t*>(sm.p1.dense)[b] = 0;
                        dense_clean = true;
                        __syncwarp();
                    }
                    if (!dirty) ic = P.coords[slot];          // (pass 1 keeps coordinates in global memory: only merges touch them)
                    else {                                   // clear the previous dense copy of this item (hs still holds its bins)
                        for (int r = lane; r < mj.nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = 0;
                        __syncwarp();
                    }
                    merge_pixels_warp<false>(ipx, P.windows + (int64_t)(base + fm) * ws, ws, P.npx);
                    const int4 kc = P.coords[base + fm];
                    ic = make_int4((ic.x + kc.x) >> 1, (ic.y + kc.y) >> 1, (ic.z + kc.z) >> 1, (ic.w + kc.w) >> 1);   // Python // (coords >= 0)
                    __syncwarp();
                    const int nnz = hist_build_warp<CAP>(ipx, P.npx, lut, sm.p1.hs, ient, P.meta + slot, sm.p1.eg, 1);
                    for (int r = lane; r < nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = (uint16_t)sm.p1.hs.cnt[r];
                    __syncwarp();
                    mj = load_meta_cg(P.meta + slot);
                    if (lane == 0) sm.hash[j] = mj.hash;     // the rebuild hashes the new pixels
                    if (lane < kHistGroups) P.E_T[(int64_t)lane * P.e_stride + slot] = sm.p1.eg[lane];   // later merges prune against the NEW histogram
                    // re-classify the updated item against the survivors after the merge position
                    scan = lane < L ? 0u : (lane == L ? (bit == 31 ? 0u : ~((2u << bit) - 1)) : 0xffffffffu);
                    fold_classify_against<RMAX, CAP>(sm, P, mj, base, A & scan, L, (j - 1) >> 5);
                    if (lane >= L && lane <= ((j - 1) >> 5)) { vd = sm.p1.rowd[lane]; vm = sm.p1.rowm[lane]; }
                    __syncwarp();
                    dirty = true;
                }
                if (dirty) {
                    if (lane == 0) P.coords[slot] = ic;
                    // the item is final: its class against every LATER item (their bit rows described the un-merged histogram)
                    const unsigned bitj = 1u << (j & 31);
                    {
                        unsigned later = 0;                  // items after j: lane w covers 32w..32w+31
                        if (lane >= (j >> 5) && lane < nwords) {
                            later = 0xffffffffu;
                            if (lane == (j >> 5)) later = (j & 31) == 31 ? 0u : ~((2u << (j & 31)) - 1);
                            if (lane == nwords - 1 && (n & 31)) later &= (1u << (n & 31)) - 1;
                        }
                        fold_classify_against<RMAX, CAP>(sm, P, mj, base, later, j >> 5, nwords - 1);
                        for (int t = j >> 5; t < nwords; t++) {
                            const int q2 = 32 * t + lane;
                            if (q2 > j && q2 < n) {
                                uint32_t* r = M + (int64_t)(base + q2) * 2 * RW + (j >> 5);
                                r[0] = (r[0] & ~bitj) | (((sm.p1.rowd[t] >> lane) & 1u) ? bitj : 0u);      // (this warp is the only writer of the frame's rows)
                                r[RW] = (r[RW] & ~bitj) | (((sm.p1.rowm[t] >> lane) & 1u) ? bitj : 0u);
                            }
                        }
                    }
                    __syncwarp();
                    for (int r = lane; r < mj.nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = 0;
                    __syncwarp();
                    if (j + 1 < n && lane < RW) { nd = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + lane); nm = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + RW + lane); }
                }
                if (__any_sync(0xffffffffu, D != 0)) A = fold_apply_deletions<RMAX, CAP>(A, D, sm, P.windows, base, ws);
                if (lane == (j >> 5)) A |= 1u << (j & 31);
            }
        } else {
            if (lane < nwords) A = (lane == nwords - 1 && (n & 31)) ? ((1u << (n & 31)) - 1) : 0xffffffffu;
        }
        if (P.do_coords) A = fold_coord_pass<RMAX, CAP>(A, sm, P, base, n, sim_cut);
        fold_emit_survivors(A, P, f, base);
        __syncwarp();
    }
}


// =====================================================================================================================
// The fold of a LARGE frame (more than kFoldCtaMin windows, at most 1024): one CTA per frame.  Warp 0 is the sequencer -- it runs
// exactly the item loop of k5_fold_warp (bit set of survivors, delete / merge bit rows, pop-by-pixel-equality) -- and the other
// warps join it for the only expensive step, the re-classification of a merged item against hundreds of other items
// (Cauchy-Schwarz pruning of 32 items per warp step, then the exact integer dots of the surviving candidates, one candidate per
// warp step) and for the rewrite of the item's column in the later items' bit rows.  A 4K frame with 2000 candidates keeps ~800
// windows after the aspect filter and merges ~100 times; with one warp per frame each merge cost ~100 us of exposed L2 latency.
// =====================================================================================================================
constexpr int kFoldCtaWarps = 8;
constexpr int kFoldCtaMin = 256;                        // frames above this size come here (the warp fold keeps the smaller ones: 126 registers x 256 threads allow only 2 such CTAs per SM)

template <int CAP>
struct FoldCtaSmem {
    HsvLut lut;
    FoldWarpSmem<1024, CAP> w;
    WinMeta mj;                  // the merged item's moments
    uint32_t cmask[32];          // items to classify against (word t = items 32t .. 32t+31); pass 2: the survivors so far
    int32_t cmd, w0, w1, ncand, frame, rewrite_j;
    uint32_t cd[32], cm[32];     // pass 2: delete / merge bits of the current item against survivor word t
    int4 ic;                     // pass 2: the current item's (possibly merged) coordinates
    int32_t start, go;           // pass 2: first list position still to scan / another round needed
};
enum { kCtaCmdClassify = 1, kCtaCmdNextFrame = 2, kCtaCmdExit = 3 };

// All warps of the CTA.  Classes of the merged item (dense histogram in w.p1.dense, moments S.mj, energies w.p1.eg) against the items
// in S.cmask words [S.w0, S.w1] -> bit words w.p1.rowd / w.p1.rowm.  With S.rewrite_j >= 0 the bits then replace column rewrite_j of
// the later items' rows of M.  Four block barriers, the same for every warp.
template <int CAP>
__device__ __forceinline__ void fold_cta_classify(FoldCtaSmem<CAP>& S, const FoldParams& P, uint32_t* M, int RW, int base, int n) {
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    FoldWarpSmem<1024, CAP>& sm = S.w;
    if (tid < 32) { sm.p1.rowd[tid] = 0; sm.p1.rowm[tid] = 0; }
    if (tid == 0) S.ncand = 0;
    __syncthreads();
    const WinMeta mj = S.mj;
    const int w0 = S.w0, w1 = S.w1;
    uint32_t* cand = sm.p1.cand();
    for (int t = w0 + wid; t <= w1; t += kFoldCtaWarps) {
        const unsigned aw = S.cmask[t];
        if (!aw) continue;
        const bool mine = (aw >> lane) & 1u;
        const int q = base + 32 * t + lane;
        int c = 0, nnz_q = 0;
        bool need = false;
        if (mine) {
            float ub = 0.f;
#pragma unroll
            for (int g = 0; g < kHistGroups; g++) ub += sm.p1.eg[g] * P.E_T[(int64_t)g * P.e_stride + q];
            const WinMeta mq = load_meta_cg(P.meta + q);
            nnz_q = mq.nnz;
            const double den2 = mj.A * mq.A;
            if (!(fabs(den2) > DBL_EPSILON)) c = classify(1.0, P.hist_tol, P.hist_lo);      // compareHist's degenerate branch
            else need = !prunable(ub, mj, mq.s1, mq.A, mq.rA, P.hist_lo);
        }
        const unsigned nb = __ballot_sync(0xffffffffu, need);
        int pos = 0;
        if (nb && lane == 0) pos = atomicAdd(&S.ncand, __popc(nb));
        pos = __shfl_sync(0xffffffffu, pos, 0);
        if (need) cand[pos + __popc(nb & ((1u << lane) - 1))] = (uint32_t)(32 * t + lane) | ((uint32_t)nnz_q << 16);
        const unsigned bd = __ballot_sync(0xffffffffu, c == 1), bm = __ballot_sync(0xffffffffu, c == 2);
        if (lane == 0) { if (bd) atomicOr(&sm.p1.rowd[t], bd); if (bm) atomicOr(&sm.p1.rowm[t], bm); }
    }
    __syncthreads();
    // exact integer dots: candidate k of a round goes to warp k % kFoldCtaWarps, slot k / kFoldCtaWarps of that warp (two in flight)
    const int ncand = S.ncand;
    const uint16_t* dense = sm.p1.dense;
    const uint4* ent4 = reinterpret_cast<const uint4*>(P.entries) + (int64_t)base * (P.es >> 2);
    const int es4 = P.es >> 2;
    for (int r0 = 0; r0 < ncand; r0 += 32 * kFoldCtaWarps) {
        const int left = ncand - r0 - wid;
        const int nr = left <= 0 ? 0 : min(32, (left + kFoldCtaWarps - 1) / kFoldCtaWarps);       // this warp's candidates of the round
        int Ik = 0;
        int cA = 0, cB = 0, nA = 0, nB = 0;
        const uint4 *eA = ent4, *eB = ent4;
        uint4 a0, a1, b0, b1;
#define CTA_FETCH(CI, N, E, V0, V1)                                                                          \
        do {                                                                                                 \
            const uint32_t info = cand[r0 + (CI) * kFoldCtaWarps + wid];                                     \
            N = (int)((info >> 16) + 3) >> 2;                                                                \
            E = ent4 + (int64_t)(info & 0xffffu) * es4;                                                      \
            V0 = lane < N ? E[lane] : make_uint4(0, 0, 0, 0);                                                \
            V1 = lane + 32 < N ? E[lane + 32] : make_uint4(0, 0, 0, 0);                                      \
        } while (0)
#define CTA_DOT(V) ((int)dense[(V).x >> 16] * (int)((V).x & 0xffffu) + (int)dense[(V).y >> 16] * (int)((V).y & 0xffffu) + \
                    (int)dense[(V).z >> 16] * (int)((V).z & 0xffffu) + (int)dense[(V).w >> 16] * (int)((V).w & 0xffffu))
#define CTA_COMPUTE(CI, N, E, V0, V1)                                                                        \
        do {                                                                                                 \
            int acc = CTA_DOT(V0) + CTA_DOT(V1);                                                             \
            for (int e = lane + 64; e < N; e += 32) { const uint4 v = E[e]; acc += CTA_DOT(v); }             \
            acc = warp_sum_i(acc);                                                                           \
            if (lane == (CI)) Ik = acc;                                                                      \
        } while (0)
        if (nr > 0) {
            CTA_FETCH(cA, nA, eA, a0, a1);
            while (cA < nr) {
                cB = cA + 1;
                if (cB < nr) CTA_FETCH(cB, nB, eB, b0, b1);
                CTA_COMPUTE(cA, nA, eA, a0, a1);
                if (cB >= nr) break;
                cA = cB + 1;
                if (cA < nr) CTA_FETCH(cA, nA, eA, a0, a1);
                CTA_COMPUTE(cB, nB, eB, b0, b1);
            }
        }
#undef CTA_FETCH
#undef CTA_DOT
#undef CTA_COMPUTE
        if (lane < nr) {                                     // lane-parallel classification (exact f64 only within 2e-6 of a threshold)
            const int ql = (int)(cand[r0 + lane * kFoldCtaWarps + wid] & 0xffffu), q = base + ql;
            const WinMeta mq = load_meta_cg(P.meta + q);
            int c = classify_from_int(Ik, mj, mq, P.hist_tol, P.hist_lo);
            if (c == kClsUnsure) {
                atomicAdd(&g_unsure_pairs, 1ull);
                const uint32_t* eo = P.entries + (int64_t)q * P.es;
                double s12 = 0;
                for (int i = 0; i < mq.nnz; i++) {
                    const uint32_t v = eo[i];
                    s12 += (double)((float)dense[v >> 16] * mj.a) * (double)((float)(v & 0xffffu) * mq.a);
                }
                c = classify(correl_from(s12, mj.s1, mj.A, mq.s1, mq.A), P.hist_tol, P.hist_lo);
            }
            if (c == 1) atomicOr(&sm.p1.rowd[ql >> 5], 1u << (ql & 31));
            else if (c == 2) atomicOr(&sm.p1.rowm[ql >> 5], 1u << (ql & 31));
        }
        __syncwarp();
    }
    __syncthreads();
    const int j = S.rewrite_j;
    if (j >= 0) {                                            // the item is final: its column in the bit rows of every LATER item
        const unsigned bitj = 1u << (j & 31);
        const int nwords = (n + 31) >> 5;
        for (int t = (j >> 5) + wid; t < nwords; t += kFoldCtaWarps) {
            const int q2 = 32 * t + lane;
            if (q2 > j && q2 < n) {
                uint32_t* r = M + (int64_t)(base + q2) * 2 * RW + (j >> 5);
                r[0] = (r[0] & ~bitj) | (((sm.p1.rowd[t] >> lane) & 1u) ? bitj : 0u);      // (this CTA is the only writer of the frame's rows)
                r[RW] = (r[RW] & ~bitj) | (((sm.p1.rowm[t] >> lane) & 1u) ? bitj : 0u);
            }
        }
    }
    __syncthreads();
}


// Pass 2 (corner similarity) of a large frame by the whole CTA: same semantics as fold_coord_pass, but the classes of the current
// item against the survivors so far (up to 32 words of 32) are computed by all warps at once, one word per warp step, instead of
// word after word by one warp -- with ~480 pass-1 survivors that scan was 40 % of the frame's fold time.  Warp 0 keeps the survivor
// set A2, finds the first merge in list order, applies merges and deletions; returns the survivors (valid in warp 0).
template <int CAP>
__device__ __forceinline__ unsigned fold_cta_coord_pass(FoldCtaSmem<CAP>& S, const FoldParams& P, int base, int n, int sim_cut, unsigned A1) {
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    FoldWarpSmem<1024, CAP>& sm = S.w;
    const int nwords = (n + 31) >> 5;
    const int ws = P.ws;
    const double tol = P.coord_tol, lo = P.coord_lo;
    for (int p = tid; p < n; p += blockDim.x) sm.coords[p] = P.coords[base + p];      // overlays the pass-1 workspace
    if (wid == 0) { S.cmask[lane] = 0; S.cd[lane] = A1; }   // cd doubles as the carrier of A1 for the other warps' item loop
    __syncthreads();
    const unsigned a1w = S.cd[lane];                         // every warp walks the same item sequence
    unsigned A2 = 0;
    __syncthreads();
    for (int tj = 0; tj < nwords; tj++) {
        unsigned wj = __shfl_sync(0xffffffffu, a1w, tj);
        while (wj) {
            const int j = 32 * tj + __ffs(wj) - 1;
            wj &= wj - 1;
            if (tid == 0) { S.ic = sm.coords[j]; S.start = 0; }
            unsigned D = 0;
            bool dirty = false;
            __syncthreads();
            while (true) {
                const int4 ic = S.ic;
                const int start = S.start;
                for (int t = (start >> 5) + wid; t <= tj; t += kFoldCtaWarps) {
                    unsigned aw = S.cmask[t];
                    if (t == (start >> 5)) aw &= ~((1u << (start & 31)) - 1);
                    int c = 0;
                    if ((aw >> lane) & 1u) c = classify(coord_sim(ic, sm.coords[32 * t + lane], P.simtab, sim_cut), tol, lo);
                    const unsigned bd = __ballot_sync(0xffffffffu, c == 1), bmm = __ballot_sync(0xffffffffu, c == 2);
                    if (lane == 0) { S.cd[t] = bd; S.cm[t] = bmm; }
                }
                __syncthreads();
                if (wid == 0) {
                    const bool in_range = lane >= (start >> 5) && lane <= tj;
                    const unsigned mw = in_range ? S.cm[lane] : 0u, dw = in_range ? S.cd[lane] : 0u;
                    const unsigned any = __ballot_sync(0xffffffffu, mw != 0u);
                    if (!any) {
                        D |= dw;
                        if (lane == 0) S.go = 0;
                    } else {
                        // ---- merge with the first survivor in the merge band (DET:217-221): pixels, coords; later comparisons use the updated item
                        const int t = __ffs(any) - 1;
                        const int bit = __ffs(__shfl_sync(0xffffffffu, mw, t)) - 1, fm = 32 * t + bit;
                        if (lane < t) D |= dw;
                        else if (lane == t) D |= (dw & ((1u << bit) - 1)) | (1u << bit);
                        const uint32_t hsh = merge_pixels_warp<true>(P.windows + (int64_t)(base + j) * ws, P.windows + (int64_t)(base + fm) * ws, ws, P.npx);
                        const int4 kc = sm.coords[fm];
                        if (lane == 0) {
                            S.ic = make_int4((ic.x + kc.x) >> 1, (ic.y + kc.y) >> 1, (ic.z + kc.z) >> 1, (ic.w + kc.w) >> 1);
                            sm.hash[j] = hsh;
                            S.start = fm + 1;
                            S.go = 1;
                        }
                        dirty = true;
                    }
                }
                __syncthreads();
                if (!S.go) break;
            }
            if (wid == 0) {
                if (dirty) {
                    if (lane == 0) { const int4 icn = S.ic; sm.coords[j] = icn; P.coords[base + j] = icn; P.meta[base + j].hash = sm.hash[j]; }
                    __syncwarp();
                }
                if (__any_sync(0xffffffffu, D != 0)) A2 = fold_apply_deletions<1024, CAP>(A2, D, sm, P.windows, base, ws);
                if (lane == (j >> 5)) A2 |= 1u << (j & 31);
                S.cmask[lane] = A2;
            }
            __syncthreads();
        }
    }
    return A2;
}

template <int CAP>
__global__ void __launch_bounds__(kFoldCtaWarps * 32) k5_fold_cta_kernel(FoldParams P, int nframes, uint32_t* M, int RW, int sim_cut,
                                                                          const int32_t* __restrict__ order, int32_t* counter, int n_skip) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    FoldCtaSmem<CAP>& S = *reinterpret_cast<FoldCtaSmem<CAP>*>(smem_raw);
    FoldWarpSmem<1024, CAP>& sm = S.w;
    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
    load_hsv_lut(S.lut, P.tab);
    const int ws = P.ws, es = P.es;
    while (true) {
        __syncthreads();                                     // (the previous frame is complete; lut loaded)
        if (tid == 0) {
            int f = -1;
            while (true) {                                   // next frame of this kernel's size class, longest first
                const int idx = atomicAdd(counter, 1);
                if (idx >= nframes) break;
                const int fc = order[idx], nc = P.offsets[fc + 1] - P.offsets[fc];
                if (nc <= 1024 && nc <= RW * 32 && nc > n_skip) { f = fc; break; }
            }
            S.frame = f;
        }
        __syncthreads();
        const int f = S.frame;
        if (f < 0) break;
        const int base = P.offsets[f], n = P.offsets[f + 1] - base;
        for (int p = tid; p < n; p += blockDim.x) sm.hash[p] = P.meta[base + p].hash;
        for (int b = tid; b < kDenseLen / 2; b += blockDim.x) reinterpret_cast<uint32_t*>(sm.p1.dense)[b] = 0;
        __syncthreads();
        if (wid != 0) {                                      // helper warps: wait for the sequencer's orders
            while (true) {
                __syncthreads();
                const int cmd = S.cmd;
                if (cmd != kCtaCmdClassify) break;
                fold_cta_classify<CAP>(S, P, M, RW, base, n);
            }
            if (P.do_coords) fold_cta_coord_pass<CAP>(S, P, base, n, sim_cut, 0u);
            continue;
        }
        // ---- warp 0: the sequencer (same item loop as k5_fold_warp) ----
        const int nwords = (n + 31) >> 5;
        unsigned A = 0;
        if (P.do_hist) {
            const uint32_t* Mf = M + (int64_t)base * 2 * RW;
            unsigned nd = 0, nm = 0;
            if (n > 1 && lane < RW) { nd = __ldcg(Mf + 2 * RW + lane); nm = __ldcg(Mf + 3 * RW + lane); }
            if (n > 0 && lane == 0) A = 1u;
            for (int j = 1; j < n; j++) {
                unsigned vd = nd, vm = nm;
                if (j + 1 < n && lane < RW) { nd = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + lane); nm = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + RW + lane); }
                unsigned D = 0, scan = 0xffffffffu;
                bool dirty = false;
                int4 ic = make_int4(0, 0, 0, 0);
                WinMeta mj;
                mj.nnz = 0;
                const int slot = base + j;
                while (true) {
                    const unsigned m = vm & A & scan, d = vd & A & scan;
                    const unsigned bm = __ballot_sync(0xffffffffu, m != 0);
                    if (!bm) { D |= d; break; }
                    // ---- merge with the first survivor (list order) in the merge band (DET:217-221) ----
                    const int L = __ffs(bm) - 1;
                    const int bit = __ffs(__shfl_sync(0xffffffffu, m, L)) - 1;
                    const int fm = 32 * L + bit;
                    if (lane < L) D |= d;
                    else if (lane == L) D |= (d & ((1u << bit) - 1)) | (1u << bit);
                    uint8_t* ipx = P.windows + (int64_t)slot * ws;
                    uint32_t* ient = P.entries + (int64_t)slot * es;
                    if (!dirty) ic = P.coords[slot];
                    else {                                   // clear the previous dense copy of this item (hs still holds its bins)
                        for (int r = lane; r < mj.nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = 0;
                        __syncwarp();
                    }
                    merge_pixels_warp<false>(ipx, P.windows + (int64_t)(base + fm) * ws, ws, P.npx);
                    const int4 kc = P.coords[base + fm];
                    ic = make_int4((ic.x + kc.x) >> 1, (ic.y + kc.y) >> 1, (ic.z + kc.z) >> 1, (ic.w + kc.w) >> 1);   // Python // (coords >= 0)
                    __syncwarp();
                    const int nnz = hist_build_warp<CAP>(ipx, P.npx, S.lut, sm.p1.hs, ient, P.meta + slot, sm.p1.eg, 1);
                    for (int r = lane; r < nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = (uint16_t)sm.p1.hs.cnt[r];
                    __syncwarp();
                    mj = load_meta_cg(P.meta + slot);
                    if (lane == 0) sm.hash[j] = mj.hash;
                    if (lane < kHistGroups) P.E_T[(int64_t)lane * P.e_stride + slot] = sm.p1.eg[lane];   // later merges prune against the NEW histogram
                    // re-classify the updated item against the survivors after the merge position (all warps)
                    scan = lane < L ? 0u : (lane == L ? (bit == 31 ? 0u : ~((2u << bit) - 1)) : 0xffffffffu);
                    S.cmask[lane] = A & scan;
                    if (lane == 0) { S.mj = mj; S.w0 = L; S.w1 = (j - 1) >> 5; S.rewrite_j = -1; S.cmd = kCtaCmdClassify; }
                    __syncthreads();
                    fold_cta_classify<CAP>(S, P, M, RW, base, n);
                    if (lane >= L && lane <= ((j - 1) >> 5)) { vd = sm.p1.rowd[lane]; vm = sm.p1.rowm[lane]; }
                    __syncwarp();
                    dirty = true;
                }
                if (dirty) {
                    if (lane == 0) P.coords[slot] = ic;
                    // the item is final: its class against every LATER item (their bit rows described the un-merged histogram)
                    unsigned later = 0;                      // items after j: lane w covers 32w..32w+31
                    if (lane >= (j >> 5) && lane < nwords) {
                        later = 0xffffffffu;
                        if (lane == (j >> 5)) later = (j & 31) == 31 ? 0u : ~((2u << (j & 31)) - 1);
                        if (lane == nwords - 1 && (n & 31)) later &= (1u << (n & 31)) - 1;
                    }
                    S.cmask[lane] = later;
                    if (lane == 0) { S.mj = mj; S.w0 = j >> 5; S.w1 = nwords - 1; S.rewrite_j = j; S.cmd = kCtaCmdClassify; }
                    __syncthreads();
                    fold_cta_classify<CAP>(S, P, M, RW, base, n);
                    for (int r = lane; r < mj.nnz; r += 32) sm.p1.dense[sm.p1.hs.binof[r]] = 0;
                    __syncwarp();
                    if (j + 1 < n && lane < RW) { nd = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + lane); nm = __ldcg(Mf + (int64_t)(j + 1) * 2 * RW + RW + lane); }
                }
                if (__any_sync(0xffffffffu, D != 0)) A = fold_apply_deletions<1024, CAP>(A, D, sm, P.windows, base, ws);
                if (lane == (j >> 5)) A |= 1u << (j & 31);
            }
        } else {
            if (lane < nwords) A = (lane == nwords - 1 && (n & 31)) ? ((1u << (n & 31)) - 1) : 0xffffffffu;
        }
        if (lane == 0) S.cmd = kCtaCmdNextFrame;             // the helpers leave their command loop and join pass 2
        __syncthreads();
        if (P.do_coords) A = fold_cta_coord_pass<CAP>(S, P, base, n, sim_cut, A);
        fold_emit_survivors(A, P, f, base);
    }
}

}  // namespace tsd
