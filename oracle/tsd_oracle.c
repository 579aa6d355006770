/*
 * tsd_oracle.c -- CPU restatement (plain C99) of the reference's candidate-window scoring and
 * recognition path.  TEST INFRASTRUCTURE ONLY: it is the checker the CUDA path is compared with
 * (tests/, __graft_entry__.smoke(), bench.py's cpu_baseline leg).  Nothing on the product path may
 * link, import or call it.
 *
 * The reference (cfkr-dev/OpenCV-Traffic-Sign-Detector) is pure Python; the arithmetic of this path
 * lives in third-party wheels that are NOT under /root/reference and are not pinned by the reference
 * (no requirements file).  De-facto pins = the versions in this image:
 *     opencv-python 4.13.0, scikit-learn 1.9.0, scipy 1.18.1, numpy 2.3.5
 * Each function below restates the published algorithm of the routine the reference calls and cites
 * the reference call site (DET = "Deteción de Objetos", REC = "Reconocimiento de Objetos").
 *
 * Pinning: the reference holds no tests / golden vectors for this path (SURVEY.md section 4), so this
 * oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF run in the build container
 * (tests/golden/make_golden.py -> tests/golden/ *.npz) and, where cv2 is importable, against live cv2.
 *
 * Build: make -C oracle   (gcc -O2 -ffp-contract=off; no FMA contraction so f64/f32 steps round
 * exactly as the reference's numpy / OpenCV scalar code does).
 */
#include <math.h>
#include <float.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------------
 * A.1  makeWindowBiggerOrDiscardFakeDetections  -- DET/source.py:155-174 (= REC/source.py:88-107)
 * box = numpy int32 (x, y, w, h); percentage = Python float literal (1.30 det / 1.15 rec).
 * Returns 1 and writes (x1,y1,x2,y2) when aspect_lo < w/h < aspect_hi (strict; the reference's 0.8 and 1.20), else 0.
 * ---------------------------------------------------------------------------------------------- */
ORC_API int orc_expand_box(int32_t x, int32_t y, int32_t w, int32_t h, double percentage, double aspect_lo, double aspect_hi,
                           int32_t out[4])
{
    double pm1 = percentage - 1.0;                 /* (percentage - 1) evaluated in f64, :161 */
    double dw = ((double)w * pm1) * 0.5;           /* w * (p-1) * 0.5, left to right          */
    double dh = ((double)h * pm1) * 0.5;
    double ratio = (double)w / (double)h;          /* numpy int32 / int32 -> float64 (:164); h==0 -> inf/nan -> reject */
    if (!(aspect_lo < ratio && ratio < aspect_hi)) return 0;
    double x1 = (double)x - dw, y1 = (double)y - dh;
    double x2 = (double)(x + w) + dw, y2 = (double)(y + h) + dh;
    x1 = x1 > 0 ? x1 : 0;  y1 = y1 > 0 ? y1 : 0;   /* only the low side is clamped (:167-168) */
    x2 = x2 > 0 ? x2 : 0;  y2 = y2 > 0 ? y2 : 0;   /* always true for valid boxes (:169-170) */
    out[0] = (int32_t)x1; out[1] = (int32_t)y1; out[2] = (int32_t)x2; out[3] = (int32_t)y2;  /* int(): trunc */
    return 1;
}

/* numpy slice clipping of image[y1:y2, x1:x2] -- DET/source.py:570-572.  coords are >= 0. */
static void clip_crop(const int32_t c[4], int H, int W, int *cx, int *cy, int *cw, int *ch)
{
    int x1 = c[0] < W ? c[0] : W, x2 = c[2] < W ? c[2] : W;
    int y1 = c[1] < H ? c[1] : H, y2 = c[3] < H ? c[3] : H;
    *cx = x1; *cy = y1; *cw = x2 > x1 ? x2 - x1 : 0; *ch = y2 > y1 ? y2 - y1 : 0;
}

/* ------------------------------------------------------------------------------------------------
 * A.2  cv2.resize(src, (D, D))  default INTER_LINEAR, uint8 -- DET/source.py:123-124, REC/source.py:57,253-254
 * OpenCV imgproc/resize.cpp: same-size copy; exact 2x in both axes -> INTER_AREA 2x2 fast path;
 * otherwise two-pass fixed point (INTER_RESIZE_COEF_BITS = 11).
 * src: h x w x C, row stride `stride` bytes.  dst: D x D x C contiguous.
 * ---------------------------------------------------------------------------------------------- */
static inline int rne_f2i(float v) { return (int)lrintf(v); }   /* cvRound: round-half-even (default FE mode) */

static void linear_coeffs(int ssize, int D, int clamp_coef, int *ofs, short *c0, short *c1)
{
    double inv_scale = (double)D / (double)ssize;
    double scale = 1.0 / inv_scale;
    for (int d = 0; d < D; d++) {
        float f = (float)(((double)d + 0.5) * scale - 0.5);
        int s = (int)floorf(f);
        f -= (float)s;
        if (clamp_coef) {                 /* X axis: coefficient clamp at the ROI edge */
            if (s < 0) { f = 0.f; s = 0; }
            if (s >= ssize - 1) { f = 0.f; s = ssize - 1; }
        }
        ofs[d] = s;
        int a = rne_f2i((1.f - f) * 2048.f), b = rne_f2i(f * 2048.f);
        c0[d] = (short)(a > 32767 ? 32767 : a);
        c1[d] = (short)(b > 32767 ? 32767 : b);
    }
}

ORC_API void orc_resize_linear_u8(const uint8_t *src, int h, int w, int stride, int C, uint8_t *dst, int D)
{
    if (h == D && w == D) {
        for (int y = 0; y < D; y++) memcpy(dst + (size_t)y * D * C, src + (size_t)y * stride, (size_t)D * C);
        return;
    }
    if (h == 2 * D && w == 2 * D) {
        for (int y = 0; y < D; y++)
            for (int x = 0; x < D; x++)
                for (int c = 0; c < C; c++) {
                    const uint8_t *p = src + (size_t)(2 * y) * stride + (size_t)(2 * x) * C + c;
                    dst[((size_t)y * D + x) * C + c] = (uint8_t)((p[0] + p[C] + p[stride] + p[stride + C] + 2) >> 2);
                }
        return;
    }
    int xo[64], yo[64]; short xa0[64], xa1[64], yb0[64], yb1[64];
    linear_coeffs(w, D, 1, xo, xa0, xa1);
    linear_coeffs(h, D, 0, yo, yb0, yb1);        /* Y axis: NO coefficient clamp; rows are clipped instead */
    for (int dy = 0; dy < D; dy++) {
        int r0 = yo[dy], r1 = yo[dy] + 1;
        r0 = r0 < 0 ? 0 : (r0 > h - 1 ? h - 1 : r0);
        r1 = r1 < 0 ? 0 : (r1 > h - 1 ? h - 1 : r1);
        const uint8_t *S0 = src + (size_t)r0 * stride, *S1 = src + (size_t)r1 * stride;
        for (int dx = 0; dx < D; dx++) {
            int s0 = xo[dx], s1 = s0 + 1 < w ? s0 + 1 : w - 1;
            for (int c = 0; c < C; c++) {
                int t0 = S0[s0 * C + c] * xa0[dx] + S0[s1 * C + c] * xa1[dx];
                int t1 = S1[s0 * C + c] * xa0[dx] + S1[s1 * C + c] * xa1[dx];
                int v = (((yb0[dy] * (t0 >> 4)) >> 16) + ((yb1[dy] * (t1 >> 4)) >> 16) + 2) >> 2;
                dst[((size_t)dy * D + dx) * C + c] = (uint8_t)v;
            }
        }
    }
}

/* crop (numpy slice, clipped to the frame) + resize -- DET/source.py:123-124.  Returns 0 if the crop is empty. */
ORC_API int orc_crop_resize(const uint8_t *frame, int H, int W, int C, const int32_t coords[4], uint8_t *dst, int D)
{
    int cx, cy, cw, ch;
    clip_crop(coords, H, W, &cx, &cy, &cw, &ch);
    if (cw <= 0 || ch <= 0) return 0;
    orc_resize_linear_u8(frame + ((size_t)cy * W + cx) * C, ch, cw, W * C, C, dst, D);
    return 1;
}

/* ------------------------------------------------------------------------------------------------
 * A.3  cv2.cvtColor(BGR2HSV) 8-bit (H in [0,180)) -- DET/source.py:65,576 (OpenCV color_hsv RGB2HSV_b,
 * hsv_shift = 12) and the inRange/add masks of getColorMaskRedOrBlue -- DET/source.py:63-89.
 * ---------------------------------------------------------------------------------------------- */
static int32_t g_sdiv[256], g_hdiv[256];
static int g_tabs_ready = 0;
static void hsv_tables(void)
{
    if (g_tabs_ready) return;
    g_sdiv[0] = g_hdiv[0] = 0;
    for (int i = 1; i < 256; i++) {
        g_sdiv[i] = (int32_t)lrint((255 << 12) / (1. * i));
        g_hdiv[i] = (int32_t)lrint((180 << 12) / (6. * i));
    }
    g_tabs_ready = 1;
}

ORC_API void orc_hsv_tables(int32_t sdiv[256], int32_t hdiv[256])
{
    hsv_tables();
    memcpy(sdiv, g_sdiv, sizeof g_sdiv); memcpy(hdiv, g_hdiv, sizeof g_hdiv);
}

static inline void bgr2hsv_px(int b, int g, int r, int *H, int *S, int *V)
{
    int v = b > g ? b : g; v = v > r ? v : r;
    int m = b < g ? b : g; m = m < r ? m : r;
    int d = v - m;
    int h;
    if (v == r) h = g - b;
    else if (v == g) h = (b - r) + 2 * d;
    else h = (r - g) + 4 * d;
    int s = (d * g_sdiv[v] + (1 << 11)) >> 12;
    h = (h * g_hdiv[d] + (1 << 11)) >> 12;       /* arithmetic shift of a possibly negative product */
    if (h < 0) h += 180;
    *H = h; *S = s; *V = v;
}

ORC_API void orc_bgr2hsv(const uint8_t *bgr, int npx, uint8_t *hsv)
{
    hsv_tables();
    for (int i = 0; i < npx; i++) {
        int H, S, V;
        bgr2hsv_px(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2], &H, &S, &V);
        hsv[3 * i] = (uint8_t)H; hsv[3 * i + 1] = (uint8_t)S; hsv[3 * i + 2] = (uint8_t)V;
    }
}

/* cv2.inRange bounds of the three bands [red band 0, red band 1, blue][H, S, V], inclusive (DET:70-87):
 * red: H in [0,10] u [160,179], S>=50, V>=10 (:70-79); blue: H in [90,128], S>=70, V>=10 (:85-87). */
static const uint8_t k_hsv_lo[9] = {0, 50, 10, 160, 50, 10, 90, 70, 10};
static const uint8_t k_hsv_hi[9] = {10, 255, 255, 179, 255, 255, 128, 255, 255};

static inline int in_band(int H, int S, int V, const uint8_t *lo, const uint8_t *hi)
{
    return H >= lo[0] && H <= hi[0] && S >= lo[1] && S <= hi[1] && V >= lo[2] && V <= hi[2];
}

/* hsv_lo / hsv_hi: uint8 [3][3] as above, or NULL for the reference's bounds */
ORC_API void orc_color_masks(const uint8_t *bgr, int npx, const uint8_t *hsv_lo, const uint8_t *hsv_hi, uint8_t *red, uint8_t *blue)
{
    hsv_tables();
    const uint8_t *lo = hsv_lo ? hsv_lo : k_hsv_lo, *hi = hsv_hi ? hsv_hi : k_hsv_hi;
    for (int i = 0; i < npx; i++) {
        int H, S, V;
        bgr2hsv_px(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2], &H, &S, &V);
        int r0 = in_band(H, S, V, lo, hi), r1 = in_band(H, S, V, lo + 3, hi + 3);
        red[i] = (uint8_t)((r0 || r1) ? 255 : 0);           /* cv2.add saturates 255+255 -> 255 */
        blue[i] = (uint8_t)(in_band(H, S, V, lo + 6, hi + 6) ? 255 : 0);
    }
}

/* ------------------------------------------------------------------------------------------------
 * A.4  calculateScoreBetweenMatrixs / getSimilarSignalType / detectionsMaskCorrelation
 *      -- DET/source.py:545-567, 248-261, 229-245.
 * mask, template in {0,255}.  matrix1 = mask*template in uint8 wraps to {0,1} (255*255 mod 256 = 1, :254),
 * matrix2 = template // 255.  Counts follow the four branches of :553-562 literally.
 * Returns the score in hundredths (Python round(x, 2) -> correctly rounded decimal of the exact double;
 * glibc "%.2f" is exactly rounded as well), or 0 in the degenerate-template case (:563-565).
 * ---------------------------------------------------------------------------------------------- */
static int round2_hundredths(double v)
{
    char buf[64];
    snprintf(buf, sizeof buf, "%.2f", v);
    return (int)lrint(strtod(buf, NULL) * 100.0);
}

ORC_API int orc_score_hundredths(const uint8_t *mask, const uint8_t *templ, int npx, int counts[4])
{
    int tp = 0, fp = 0, fn = 0, tn = 0;
    for (int i = 0; i < npx; i++) {
        uint8_t m1 = (uint8_t)(mask[i] * templ[i]);          /* uint8 wrap-around product */
        uint8_t m2 = (uint8_t)(templ[i] / 255);
        if (m1 == 1 && m2 == 1) tp++;
        else if (m1 == 1 && m2 == 0) fp++;
        else if (m1 == 0 && m2 == 1) fn++;
        else tn++;
    }
    if (counts) { counts[0] = tp; counts[1] = fp; counts[2] = fn; counts[3] = tn; }
    double shape = (double)npx;
    if (shape + shape * 0.01 >= (double)tn && (double)tn >= shape - shape * 0.01) return 0;
    return round2_hundredths((2.0 * tp) / (double)((2 * tp) + fp + fn));
}

/* getSimilarSignalType: first strict maximum over the 6 templates; id = index+1 (:248-261) */
ORC_API void orc_best_template(const uint8_t *mask, const uint8_t *templates6, int npx, int *score, int *id)
{
    int best = -1, bid = 0;                                   /* -inf start: any score (>= 0) wins first */
    for (int k = 0; k < 6; k++) {
        int s = orc_score_hundredths(mask, templates6 + (size_t)k * npx, npx, NULL);
        if (s > best) { best = s; bid = k + 1; }
    }
    *score = best; *id = bid;
}

/* detectionsMaskCorrelation (:229-245): red wins only if strictly greater; emit iff winner > tol.
 * Returns 1 and fills (id, hundredths) if emitted. tol_hundredths = 55 for 0.55. */
ORC_API int orc_score_window(const uint8_t *bgr, int D, const uint8_t *red6, const uint8_t *blue6,
                             int tol_hundredths, const uint8_t *hsv_lo, const uint8_t *hsv_hi, int *id, int *hundredths)
{
    int npx = D * D;
    uint8_t *r = (uint8_t *)malloc((size_t)npx), *b = (uint8_t *)malloc((size_t)npx);
    orc_color_masks(bgr, npx, hsv_lo, hsv_hi, r, b);
    int sr, ir, sb, ib;
    orc_best_template(r, red6, npx, &sr, &ir);
    orc_best_template(b, blue6, npx, &sb, &ib);
    free(r); free(b);
    if (sr > sb) { *id = ir; *hundredths = sr; return sr > tol_hundredths; }
    *id = ib; *hundredths = sb; return sb > tol_hundredths;
}

/* ------------------------------------------------------------------------------------------------
 * A.5  calculateHistAndNormalize (DET/source.py:575-586) + cv2.compareHist CORREL (:200-202)
 * calcHist 2-D uniform on (H,S): hb = floor(H*(50/180.)), sb = floor(S*(60/256.)) (OpenCV builds the
 * per-channel LUT with exactly `cvFloor(v*a + b)`, a = histSize/(hi-lo), b = -lo*a).
 * normalize NORM_MINMAX alpha=0 beta=1 on float32: scale = (1-0)/(max-min) in f64 (0 if range <= DBL_EPSILON),
 * shift = 0 - min*scale;  convertTo: out = (float)cnt*(float)scale + (float)shift  in float32.
 * ---------------------------------------------------------------------------------------------- */
#define HB 50
#define SB 60
#define NBIN (HB * SB)

ORC_API void orc_hist_bins(int hbin[180], int sbin[256])
{
    double a_h = 50 / (180. - 0.), a_s = 60 / (256. - 0.);
    for (int i = 0; i < 180; i++) hbin[i] = (int)floor(i * a_h + (-0. * a_h));
    for (int i = 0; i < 256; i++) sbin[i] = (int)floor(i * a_s + (-0. * a_s));
}

ORC_API void orc_hist_normalized(const uint8_t *bgr, int npx, float *hist /* [3000] */)
{
    static int hbin[180], sbin[256], ready = 0;
    if (!ready) { orc_hist_bins(hbin, sbin); ready = 1; }
    hsv_tables();
    for (int i = 0; i < NBIN; i++) hist[i] = 0.f;
    for (int i = 0; i < npx; i++) {
        int H, S, V;
        bgr2hsv_px(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2], &H, &S, &V);
        hist[hbin[H] * SB + sbin[S]] += 1.f;
    }
    float mn = hist[0], mx = hist[0];
    for (int i = 1; i < NBIN; i++) { if (hist[i] < mn) mn = hist[i]; if (hist[i] > mx) mx = hist[i]; }
    double smin = mn, smax = mx;
    double scale = (1.0 - 0.0) * ((smax - smin) > DBL_EPSILON ? 1. / (smax - smin) : 0.);
    double shift = 0.0 - smin * scale;
    float a = (float)scale, b = (float)shift;
    for (int i = 0; i < NBIN; i++) hist[i] = hist[i] * a + b;
}

ORC_API double orc_hist_correl(const float *h1, const float *h2)
{
    double s1 = 0, s2 = 0, s11 = 0, s12 = 0, s22 = 0;
    for (int j = 0; j < NBIN; j++) {
        double a = h1[j], b = h2[j];
        s12 += a * b; s1 += a; s11 += a * a; s2 += b; s22 += b * b;
    }
    double scale = 1. / NBIN;
    double num = s12 - s1 * s2 * scale;
    double denom2 = (s11 - s1 * s1 * scale) * (s22 - s2 * s2 * scale);
    return fabs(denom2) > DBL_EPSILON ? num / sqrt(denom2) : 1.;
}

/* EuclDSimilarity -- DET/source.py:459-462.  np.linalg.norm of an int vector -> sqrt(dx^2+dy^2) in f64. */
ORC_API double orc_eucl_similarity_d2(int64_t d2)
{
    if (d2 <= 0) return 1.0;
    double d = sqrt((double)d2);
    return 1.0 / (1.0 + pow(M_E, ((0.154 * pow(d, 1.2)) - 31.8) / (0.2 * d)));
}

ORC_API double orc_coord_similarity(const int32_t a[4], const int32_t b[4])
{
    int64_t dx = (int64_t)a[0] - b[0], dy = (int64_t)a[1] - b[1];
    int64_t ex = (int64_t)a[2] - b[2], ey = (int64_t)a[3] - b[3];
    return sqrt(orc_eucl_similarity_d2(dx * dx + dy * dy) * orc_eucl_similarity_d2(ex * ex + ey * ey));
}

/* cv2.addWeighted(a, .5, b, .5, 0) on uint8 -- DET/source.py:219: (a+b)/2 exactly representable in f32,
 * saturate_cast<uchar> = round-half-even. */
static inline uint8_t avg_rne(uint8_t a, uint8_t b)
{
    int s = a + b;
    return (uint8_t)((s >> 1) + ((s & 1) & ((s >> 1) & 1)));
}

/* cleanDuplicatedDetections -- DET/source.py:177-189 with checkIfImageIsDuplicatedOrMergeSimilarOnes :192-223,
 * getElementIndexFromList :471-477, meanCoords :465-468.
 * windows: n x (D*D*3) uint8 (in place: survivors are compacted to the front, in list order)
 * coords : n x 4 int32.   by_coords = 0: histogram CORREL similarity; 1: corner-distance similarity.
 * Returns number of survivors.  stats (optional, int[3]) += {comparisons, deletions, merges}. */
ORC_API int orc_dedup(uint8_t *windows, int32_t *coords, int n, int D, int by_coords, double tol, double merge_factor,
                      int64_t *stats)
{
    size_t wb = (size_t)D * D * 3;
    int npx = D * D;
    uint8_t *clean_px = (uint8_t *)malloc(wb * (size_t)(n > 0 ? n : 1));
    int32_t *clean_co = (int32_t *)malloc(sizeof(int32_t) * 4 * (size_t)(n > 0 ? n : 1));
    float *clean_h = by_coords ? NULL : (float *)malloc(sizeof(float) * NBIN * (size_t)(n > 0 ? n : 1));
    int *del = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
    uint8_t *del_px = (uint8_t *)malloc(wb * (size_t)(n > 0 ? n : 1));
    uint8_t *item = (uint8_t *)malloc(wb);
    float *item_h = (float *)malloc(sizeof(float) * NBIN);
    int nc = 0;
    double lo = tol * merge_factor;
    for (int i = 0; i < n; i++) {
        int32_t ic[4];
        memcpy(item, windows + wb * i, wb);
        memcpy(ic, coords + 4 * i, sizeof ic);
        if (!by_coords) orc_hist_normalized(item, npx, item_h);
        int nd = 0;
        for (int k = 0; k < nc; k++) {
            double sim = by_coords ? orc_coord_similarity(ic, clean_co + 4 * k) : orc_hist_correl(item_h, clean_h + (size_t)NBIN * k);
            if (stats) stats[0]++;
            if (sim > tol) {
                del[nd++] = k;
            } else if (lo <= sim && sim <= tol) {
                const uint8_t *q = clean_px + wb * k;
                for (size_t t = 0; t < wb; t++) item[t] = avg_rne(item[t], q[t]);
                for (int t = 0; t < 4; t++) {          /* Python // on non-negative ints */
                    int64_t s = (int64_t)ic[t] + clean_co[4 * k + t];
                    ic[t] = (int32_t)(s >= 0 ? s / 2 : -((-s + 1) / 2));
                }
                if (!by_coords) orc_hist_normalized(item, npx, item_h);
                del[nd++] = k;
                if (stats) stats[2]++;
            }
        }
        /* pop, for each deletion in order, the FIRST live entry whose pixels equal the deleted one's */
        for (int t = 0; t < nd; t++) memcpy(del_px + wb * t, clean_px + wb * del[t], wb);
        for (int t = 0; t < nd; t++) {
            int idx = -1;
            for (int k = 0; k < nc; k++)
                if (memcmp(clean_px + wb * k, del_px + wb * t, wb) == 0) { idx = k; break; }
            if (idx < 0) continue;                      /* cannot happen: the deleted entry itself matches */
            memmove(clean_px + wb * idx, clean_px + wb * (idx + 1), wb * (size_t)(nc - idx - 1));
            memmove(clean_co + 4 * idx, clean_co + 4 * (idx + 1), sizeof(int32_t) * 4 * (size_t)(nc - idx - 1));
            if (!by_coords) memmove(clean_h + (size_t)NBIN * idx, clean_h + (size_t)NBIN * (idx + 1), sizeof(float) * NBIN * (size_t)(nc - idx - 1));
            nc--;
            if (stats) stats[1]++;
        }
        memcpy(clean_px + wb * nc, item, wb);
        memcpy(clean_co + 4 * nc, ic, sizeof ic);
        if (!by_coords) memcpy(clean_h + (size_t)NBIN * nc, item_h, sizeof(float) * NBIN);
        nc++;
    }
    memcpy(windows, clean_px, wb * (size_t)nc);
    memcpy(coords, clean_co, sizeof(int32_t) * 4 * (size_t)nc);
    free(clean_px); free(clean_co); free(clean_h); free(del); free(del_px); free(item); free(item_h);
    return nc;
}

/* ------------------------------------------------------------------------------------------------
 * A.6  cv2.cvtColor(BGR2GRAY) uint8 -- REC/source.py:388 (and frame-level :254)
 * ---------------------------------------------------------------------------------------------- */
ORC_API void orc_bgr2gray(const uint8_t *bgr, int npx, uint8_t *gray)
{
    for (int i = 0; i < npx; i++)
        gray[i] = (uint8_t)((3735 * bgr[3 * i] + 19235 * bgr[3 * i + 1] + 9798 * bgr[3 * i + 2] + 16384) >> 15);
}

/* ------------------------------------------------------------------------------------------------
 * N1  grayAndEnhanceContrast -- DET/source.py:135-152 (= REC/source.py:67-84), gammaCorrection :599-605.
 *     cv2.cvtColor(BGR2GRAY) (A.6) -> cv2.createCLAHE(clipLimit=2).apply -> cv2.GaussianBlur((3,3), 0) -> cv2.LUT(gamma).
 *     OpenCV imgproc/clahe.cpp: 8x8 tiles (the image is extended to a multiple of the grid with BORDER_REFLECT_101 for
 *     the tile histograms only), clip = max(int(clipLimit * tileArea / 256), 1), excess redistributed (batch + stride),
 *     LUT = cvRound(cumsum * (255f / tileArea)), per pixel float bilinear blend of the 4 neighbouring tile LUTs in the
 *     order (l11*xa1 + l12*xa)*ya1 + (l21*xa1 + l22*xa)*ya, cvRound.  GaussianBlur 3x3 sigma 0 on 8U = exact
 *     (1 2 1)x(1 2 1)/16 with round-half-up, BORDER_REFLECT_101.  0 mismatches against cv2 4.13.0 on real frames, noise,
 *     4K and sizes that are not multiples of 8.
 * ---------------------------------------------------------------------------------------------- */
static int reflect101(int i, int n) { if (n == 1) return 0; while (i < 0 || i >= n) i = i < 0 ? -i : 2 * n - 2 - i; return i; }

ORC_API void orc_clahe(const uint8_t *src, int H, int W, double clip_limit, int tiles_x, int tiles_y, uint8_t *dst)
{
    /* clahe.cpp: when EITHER size is not a multiple of the grid, copyMakeBorder pads bottom by tilesY - rows % tilesY and right
     * by tilesX - cols % tilesX -- i.e. a whole extra grid step on the axis that WAS a multiple */
    int divisible = H % tiles_y == 0 && W % tiles_x == 0;
    int He = divisible ? H : H + tiles_y - H % tiles_y, We = divisible ? W : W + tiles_x - W % tiles_x;
    int tw = We / tiles_x, th = He / tiles_y, total = tw * th;
    float lut_scale = 255.0f / (float)total;
    int clip = 0;
    if (clip_limit > 0.0) { clip = (int)(clip_limit * total / 256); if (clip < 1) clip = 1; }
    uint8_t *lut = (uint8_t *)malloc((size_t)tiles_x * tiles_y * 256);
    for (int ty = 0; ty < tiles_y; ty++)
        for (int tx = 0; tx < tiles_x; tx++) {
            int hist[256];
            memset(hist, 0, sizeof hist);
            for (int y = ty * th; y < (ty + 1) * th; y++)
                for (int x = tx * tw; x < (tx + 1) * tw; x++) hist[src[(size_t)reflect101(y, H) * W + reflect101(x, W)]]++;
            if (clip > 0) {
                int clipped = 0;
                for (int i = 0; i < 256; i++) if (hist[i] > clip) { clipped += hist[i] - clip; hist[i] = clip; }
                int batch = clipped / 256, residual = clipped - batch * 256;
                for (int i = 0; i < 256; i++) hist[i] += batch;
                if (residual != 0) {
                    int step = 256 / residual; if (step < 1) step = 1;
                    for (int i = 0; i < 256 && residual > 0; i += step, residual--) hist[i]++;
                }
            }
            int sum = 0;
            uint8_t *l = lut + ((size_t)ty * tiles_x + tx) * 256;
            for (int i = 0; i < 256; i++) {
                sum += hist[i];
                long v = lrintf((float)sum * lut_scale);
                l[i] = (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v);
            }
        }
    float inv_tw = 1.0f / (float)tw, inv_th = 1.0f / (float)th;
    for (int y = 0; y < H; y++) {
        float tyf = (float)y * inv_th - 0.5f;
        int ty1 = (int)floorf(tyf), ty2 = ty1 + 1;
        float ya = tyf - (float)ty1, ya1 = 1.0f - ya;
        if (ty1 < 0) ty1 = 0;
        if (ty2 > tiles_y - 1) ty2 = tiles_y - 1;
        for (int x = 0; x < W; x++) {
            float txf = (float)x * inv_tw - 0.5f;
            int tx1 = (int)floorf(txf), tx2 = tx1 + 1;
            float xa = txf - (float)tx1, xa1 = 1.0f - xa;
            if (tx1 < 0) tx1 = 0;
            if (tx2 > tiles_x - 1) tx2 = tiles_x - 1;
            int v = src[(size_t)y * W + x];
            float l11 = lut[((size_t)ty1 * tiles_x + tx1) * 256 + v], l12 = lut[((size_t)ty1 * tiles_x + tx2) * 256 + v];
            float l21 = lut[((size_t)ty2 * tiles_x + tx1) * 256 + v], l22 = lut[((size_t)ty2 * tiles_x + tx2) * 256 + v];
            float res = (l11 * xa1 + l12 * xa) * ya1 + (l21 * xa1 + l22 * xa) * ya;
            long r = lrintf(res);
            dst[(size_t)y * W + x] = (uint8_t)(r < 0 ? 0 : r > 255 ? 255 : r);
        }
    }
    free(lut);
}

ORC_API void orc_gauss3(const uint8_t *src, int H, int W, uint8_t *dst)
{
    for (int y = 0; y < H; y++) {
        const uint8_t *r0 = src + (size_t)reflect101(y - 1, H) * W, *r1 = src + (size_t)y * W, *r2 = src + (size_t)reflect101(y + 1, H) * W;
        for (int x = 0; x < W; x++) {
            int xl = reflect101(x - 1, W), xr = reflect101(x + 1, W);
            int s = r0[xl] + 2 * r0[x] + r0[xr] + 2 * r1[xl] + 4 * r1[x] + 2 * r1[xr] + r2[xl] + 2 * r2[x] + r2[xr];
            dst[(size_t)y * W + x] = (uint8_t)((s + 8) >> 4);
        }
    }
}

/* the whole grayAndEnhanceContrast: gamma_table = the reference's own 256-entry table (DET/source.py:602-603) */
ORC_API void orc_preprocess(const uint8_t *bgr, int H, int W, double clip_limit, int tiles_x, int tiles_y,
                            const uint8_t *gamma_table, uint8_t *out)
{
    size_t n = (size_t)H * W;
    uint8_t *g = (uint8_t *)malloc(n), *c = (uint8_t *)malloc(n);
    orc_bgr2gray(bgr, (int)n, g);
    orc_clahe(g, H, W, clip_limit, tiles_x, tiles_y, c);
    orc_gauss3(c, H, W, g);
    for (size_t i = 0; i < n; i++) out[i] = gamma_table[g[i]];
    free(g); free(c);
}

/* ------------------------------------------------------------------------------------------------
 * A.7  cv2.HOGDescriptor(win 32x32, block 16x16, stride 8x8, cell 8x8, 9 bins, signed).compute(img)
 *      -- REC/source.py:487-494,519; REC/constants.py:14.  OpenCV objdetect/hog.cpp:
 *      computeGradient (BORDER_REFLECT_101, cartToPolar with the polynomial fastAtan), HOGCache
 *      (Gaussian window sigma = (16+16)/8 = 4 times bilinear cell votes), L2-Hys 0.2.
 * ---------------------------------------------------------------------------------------------- */
static float fast_atan_deg(float y, float x)
{
    const float scale = (float)(180.0 / M_PI);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale;
    const float p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    float ax = fabsf(x), ay = fabsf(y), a, c, c2;
    if (ax >= ay) {
        c = ay / (ax + (float)DBL_EPSILON); c2 = c * c;
        a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    } else {
        c = ax / (ay + (float)DBL_EPSILON); c2 = c * c;
        a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

#define HOG_WIN 32
#define HOG_LEN 324

ORC_API void orc_hog_32(const uint8_t *gray /* 32x32 */, float *desc /* 324 */)
{
    const int W = HOG_WIN, nb = 9;
    static float grad[HOG_WIN * HOG_WIN][2];
    static int qang[HOG_WIN * HOG_WIN][2];
    const float angleScale = (float)(nb / (2.0 * M_PI));
    for (int y = 0; y < W; y++) {
        int yp = y - 1 < 0 ? 1 : y - 1, yn = y + 1 >= W ? W - 2 : y + 1;
        for (int x = 0; x < W; x++) {
            int xp = x - 1 < 0 ? 1 : x - 1, xn = x + 1 >= W ? W - 2 : x + 1;
            float dx = (float)gray[y * W + xn] - (float)gray[y * W + xp];
            float dy = (float)gray[yn * W + x] - (float)gray[yp * W + x];
            float mag = sqrtf(dx * dx + dy * dy);
            float ang = fast_atan_deg(dy, dx) * (float)(M_PI / 180.0);
            float t = ang * angleScale - 0.5f;
            int hidx = (int)floorf(t);
            t -= (float)hidx;
            grad[y * W + x][0] = mag * (1.f - t);
            grad[y * W + x][1] = mag * t;
            if (hidx < 0) hidx += nb; else if (hidx >= nb) hidx -= nb;
            qang[y * W + x][0] = hidx;
            hidx++; if (hidx >= nb) hidx = 0;
            qang[y * W + x][1] = hidx;
        }
    }
    /* Gaussian weights: exp(-(i-8)^2/(2*4^2)) per axis, multiplied */
    float gw[16];
    { float sigma = 4.f, sc = 1.f / (sigma * sigma * 2); for (int i = 0; i < 16; i++) { float di = i - 16 * 0.5f; gw[i] = expf(-di * di * sc); } }
    for (int bx = 0; bx < 3; bx++)
        for (int by = 0; by < 3; by++) {
            float hist[36];
            for (int k = 0; k < 36; k++) hist[k] = 0.f;
            for (int j = 0; j < 16; j++)
                for (int i = 0; i < 16; i++) {
                    float cellX = (i + 0.5f) / 8 - 0.5f, cellY = (j + 0.5f) / 8 - 0.5f;
                    int ix0 = (int)floorf(cellX), iy0 = (int)floorf(cellY);
                    float fx = cellX - ix0, fy = cellY - iy0;
                    float w = gw[i] * gw[j];
                    int p = (by * 8 + j) * W + (bx * 8 + i);
                    for (int a = 0; a < 2; a++)
                        for (int b = 0; b < 2; b++) {
                            int ix = ix0 + a, iy = iy0 + b;
                            if (ix < 0 || ix >= 2 || iy < 0 || iy >= 2) continue;
                            float hw = (a ? fx : 1.f - fx) * (b ? fy : 1.f - fy);
                            float ww = w * hw;
                            float *h = hist + (ix * 2 + iy) * nb;
                            h[qang[p][0]] += grad[p][0] * ww;
                            h[qang[p][1]] += grad[p][1] * ww;
                        }
                }
            float sum = 0;
            for (int k = 0; k < 36; k++) sum += hist[k] * hist[k];
            float sc = 1.f / (sqrtf(sum) + 36 * 0.1f);
            sum = 0;
            for (int k = 0; k < 36; k++) { hist[k] = fminf(hist[k] * sc, 0.2f); sum += hist[k] * hist[k]; }
            sc = 1.f / (sqrtf(sum) + 1e-3f);
            float *o = desc + (bx * 3 + by) * 36;
            for (int k = 0; k < 36; k++) o[k] = hist[k] * sc;
        }
}

/* ------------------------------------------------------------------------------------------------
 * A.8  predictProbabilityLDAClassifiers + extractBestPredictions + noSignDetected
 *      -- REC/source.py:565-577, 627-641, 342-347.  sklearn LinearDiscriminantAnalysis.predict_proba
 *      (binary): z = X @ coef_.T + intercept_ (float64), p1 = expit(z), p0 = 1 - p1.
 * The decision below follows the reference loops literally (best = max(p0,p1) tagged 0 or c+1; no sign
 * unless some non-zero tag has best > tol; else first maximum among non-zero tags).
 * W: [324][6] row-major (feature-major), b: [6].  logits out: [n][6].
 * ---------------------------------------------------------------------------------------------- */
static double expit_d(double z) { return 1.0 / (1.0 + exp(-z)); }   /* scipy.special.expit (f64) */

ORC_API void orc_lda_predict(const float *X, int n, int nfeat, const double *W, const double *b, double tol,
                             double *logits, int32_t *labels)
{
    for (int i = 0; i < n; i++) {
        double best[6]; int tag[6];
        for (int c = 0; c < 6; c++) {
            double z = 0;
            for (int f = 0; f < nfeat; f++) z += (double)X[(size_t)i * nfeat + f] * W[(size_t)f * 6 + c];
            z += b[c];
            if (logits) logits[(size_t)i * 6 + c] = z;
            double p1 = expit_d(z), p0 = 1.0 - p1;
            best[c] = p0 > p1 ? p0 : p1;
            tag[c] = p0 > p1 ? 0 : c + 1;
        }
        int nosign = 1;
        for (int c = 0; c < 6; c++) if (tag[c] != 0 && best[c] > tol) { nosign = 0; break; }
        int lab = 0;
        if (!nosign) {
            double bv = -INFINITY; int first = 1;
            for (int c = 0; c < 6; c++) {
                double key = tag[c] != 0 ? best[c] : -INFINITY;
                if (first || key > bv) { bv = key; lab = tag[c]; first = 0; }
            }
        }
        labels[i] = lab;
    }
}

/* predictProbabilityKNNClassifiers -- REC/source.py:592-596: Z = (X - xbar_) @ scalings_[:, :6] (f64);
 * KNeighborsClassifier(4).predict: Euclidean, uniform vote, ties -> smallest label; equal distances ->
 * smaller training index (brute-force model; sklearn uses a kd-tree with identical labels, SURVEY A.8). */
ORC_API void orc_knn_predict(const float *X, int n, int nfeat, const double *xbar, const double *S /* [nfeat][6] */,
                             const double *Ztrain /* [ntrain][6] */, const int32_t *ytrain, int ntrain, int k,
                             double *Zout, int32_t *labels)
{
    for (int i = 0; i < n; i++) {
        double z[6] = {0, 0, 0, 0, 0, 0};
        for (int f = 0; f < nfeat; f++) {
            double xc = (double)X[(size_t)i * nfeat + f] - xbar[f];
            for (int c = 0; c < 6; c++) z[c] += xc * S[(size_t)f * 6 + c];
        }
        if (Zout) memcpy(Zout + (size_t)i * 6, z, sizeof z);
        double bd[16]; int bi[16]; int nb = 0;
        for (int t = 0; t < ntrain; t++) {
            double d = 0;
            for (int c = 0; c < 6; c++) { double e = z[c] - Ztrain[(size_t)t * 6 + c]; d += e * e; }
            if (nb < k || d < bd[nb - 1]) {
                int pos = nb < k ? nb : k - 1;
                while (pos > 0 && bd[pos - 1] > d) { bd[pos] = bd[pos - 1]; bi[pos] = bi[pos - 1]; pos--; }
                bd[pos] = d; bi[pos] = t;
                if (nb < k) nb++;
            }
        }
        int votes[16] = {0};
        for (int t = 0; t < nb; t++) { int y = ytrain[bi[t]]; if (y >= 0 && y < 16) votes[y]++; }
        int lab = 0, bv = -1;
        for (int y = 0; y < 16; y++) if (votes[y] > bv) { bv = votes[y]; lab = y; }
        labels[i] = lab;
    }
}

/* ------------------------------------------------------------------------------------------------
 * Whole-frame restatement of MSERTrafficSignDetector's post-MSER part (DET/source.py:116-131) followed by
 * the mask-correlation filter (:708-716); used as the bounded CPU sample in bench.py and in parity tests.
 * boxes: n x 4 (x,y,w,h).  Outputs (capacity n): det_coords [.,4], det_id, det_hundredths.
 * The tsd_config fields: aspect bounds (0.8, 1.20), HSV bounds (NULL = the reference's), hist_tol 0.85, coord_tol 0.95,
 * merge_factor 0.8823.
 * stage_counts (optional int[4]) = {raw, aspect-passing, survivors after both passes, detections}.
 * ---------------------------------------------------------------------------------------------- */
ORC_API int orc_detect_frame(const uint8_t *frame, int H, int W, const int32_t *boxes, int n, double percentage, int D,
                             const uint8_t *red6, const uint8_t *blue6, int tol_hundredths, double aspect_lo, double aspect_hi,
                             const uint8_t *hsv_lo, const uint8_t *hsv_hi, double hist_tol, double coord_tol, double merge_factor,
                             int32_t *det_coords, int32_t *det_id, int32_t *det_hundredths,
                             uint8_t *surv_windows /* optional, n*D*D*3 */, int32_t *surv_coords /* optional n*4 */,
                             int32_t *stage_counts)
{
    size_t wb = (size_t)D * D * 3;
    uint8_t *win = (uint8_t *)malloc(wb * (size_t)(n > 0 ? n : 1));
    int32_t *co = (int32_t *)malloc(sizeof(int32_t) * 4 * (size_t)(n > 0 ? n : 1));
    int m = 0;
    for (int i = 0; i < n; i++) {
        int32_t c[4];
        if (!orc_expand_box(boxes[4 * i], boxes[4 * i + 1], boxes[4 * i + 2], boxes[4 * i + 3], percentage, aspect_lo, aspect_hi, c)) continue;
        if (!orc_crop_resize(frame, H, W, 3, c, win + wb * m, D)) continue;   /* cv2.resize would raise on an empty crop */
        memcpy(co + 4 * m, c, sizeof c);
        m++;
    }
    int passing = m;
    m = orc_dedup(win, co, m, D, 0, hist_tol, merge_factor, NULL);
    m = orc_dedup(win, co, m, D, 1, coord_tol, merge_factor, NULL);
    if (surv_windows) memcpy(surv_windows, win, wb * (size_t)m);
    if (surv_coords) memcpy(surv_coords, co, sizeof(int32_t) * 4 * (size_t)m);
    int nd = 0;
    for (int i = 0; i < m; i++) {
        int id, hs;
        if (orc_score_window(win + wb * i, D, red6, blue6, tol_hundredths, hsv_lo, hsv_hi, &id, &hs)) {
            memcpy(det_coords + 4 * nd, co + 4 * i, sizeof(int32_t) * 4);
            det_id[nd] = id; det_hundredths[nd] = hs; nd++;
        }
    }
    if (stage_counts) { stage_counts[0] = n; stage_counts[1] = passing; stage_counts[2] = m; stage_counts[3] = nd; }
    free(win); free(co);
    return nd;
}
