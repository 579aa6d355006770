/*
 * tsd_b200.h -- C ABI of the B200-native candidate-window scoring and recognition path.
 *
 * The reference (cfkr-dev/OpenCV-Traffic-Sign-Detector) has no FFI: its boundary for this path is the set of
 * module-level Python functions in the two source.py files (SURVEY.md section 8(b)).  Each entry point below
 * names the reference function(s) it replaces (DET = "Deteción de Objetos/source.py",
 * REC = "Reconocimiento de Objetos/source.py"); INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types.
 *   - every function returns 0 on success, <0 on error (TSD_E_*); tsd_last_error() gives the message of the
 *     last failing call on the calling thread.  Nothing throws.
 *   - `mem` says where ALL data pointers of that call live: TSD_MEM_HOST (the library copies through its own
 *     device staging buffers, synchronously) or TSD_MEM_DEVICE (pointers are device memory of the context's GPU;
 *     work is enqueued on the context's stream and the call returns without synchronising unless it has to
 *     report a count to the host).
 *   - one context per (process, GPU); calls on one context must be serialised by the caller.
 *   - there is no CPU fallback: without a CUDA device tsd_create fails.
 *   - layouts: frames uint8 [nframes][H][W][3] BGR with `frame_stride` bytes between frames and `row_stride`
 *     bytes between rows; boxes int32 [n][4] = (x, y, w, h) as produced by cv2.MSER.detectRegions()[1];
 *     coords int32 [n][4] = (x1, y1, x2, y2); windows uint8 [n][D][D][3]; *_offsets int32 [nframes+1]
 *     (CSR: items of frame f are offsets[f] .. offsets[f+1]-1, in the reference's list order).
 */
#ifndef TSD_B200_H
#define TSD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSD_API __attribute__((visibility("default")))

#define TSD_OK 0
#define TSD_E_INVALID (-1)   /* bad argument */
#define TSD_E_CUDA (-2)      /* CUDA runtime error (message in tsd_last_error) */
#define TSD_E_STATE (-3)     /* templates / weights not set */
#define TSD_E_NOMEM (-4)

#define TSD_MEM_HOST 0
#define TSD_MEM_DEVICE 1

#define TSD_HOG_LEN 324      /* 3x3 blocks x 4 cells x 9 bins, REC/constants.py:14 */
#define TSD_NCLASS 6         /* DET/constants.py:1 SIGNALLIST */

typedef struct tsd_ctx tsd_ctx;

/* All hard-coded constants of the reference path, one POD (SURVEY.md section 5 "config / flags").  tsd_create refuses (TSD_E_INVALID)
 * a window outside 2..32 and a coord_tol * merge_factor that is not above sqrt(f(65535)) = 0.3913: pairs whose corners are further
 * apart than the 65 536-entry corner-similarity table reaches (255 px) take no action, which equals the reference only while their
 * similarity, at most sqrt(f(65535)), is below the lowest similarity that acts. */
typedef struct tsd_config {
    double enlarge;            /* 1.30 DET/source.py:119 ; 1.15 REC/source.py:54 */
    double aspect_lo;          /* 0.8  DET/source.py:164 (strict) */
    double aspect_hi;          /* 1.20 */
    int32_t window;            /* D: 25 DET/source.py:124 ; 32 REC/source.py:57 */
    int32_t score_tol_hundredths; /* 55 = 0.55, DET/source.py:712 */
    double hist_tol;           /* 0.85 DET/source.py:127 */
    double coord_tol;          /* 0.95 DET/source.py:129 */
    double merge_factor;       /* 0.8823 DET/source.py:217 */
    uint8_t red_lo[2][3];      /* HSV inRange lower bounds of the two red bands, DET/source.py:70,75 */
    uint8_t red_hi[2][3];      /* upper bounds, DET/source.py:71,76 */
    uint8_t blue_lo[3];        /* DET/source.py:85 */
    uint8_t blue_hi[3];        /* DET/source.py:86 */
    uint8_t pad_[6];
    double proba_tol;          /* 0.5 REC/source.py:761 */
    int32_t knn_k;             /* 4 REC/source.py:607 */
    int32_t reserved;
} tsd_config;

/* flavour 0 = detection (1.30 / 25), 1 = recognition (1.15 / 32). */
TSD_API int tsd_config_default(tsd_config *cfg, int flavour);

TSD_API const char *tsd_last_error(void);
TSD_API const char *tsd_version(void);
TSD_API int tsd_device_count(void);

TSD_API int tsd_create(tsd_ctx **ctx, int device, const tsd_config *cfg /* NULL -> detection defaults */);
TSD_API int tsd_destroy(tsd_ctx *ctx);
/* The context's cudaStream_t (as void*), so callers (torch) can order their own work with it. */
TSD_API void *tsd_stream(tsd_ctx *ctx);
TSD_API int tsd_synchronize(tsd_ctx *ctx);
/* Consecutive tsd_enqueue_frames calls alternate between two scratch slots and two internal streams, so the latency-bound fold
 * of one batch runs under the throughput-bound kernels of the next (TSD_OVERLAP=0 in the environment turns this off).  The
 * context's stream therefore waits for a batch only when the NEXT batch is enqueued, or when tsd_flush / tsd_synchronize /
 * tsd_fetch_detections is called: tsd_flush makes tsd_stream() wait for everything enqueued so far without blocking the host.
 * The front half of a batch (K1, K2, histograms, pair classes) starts only when the previous batch's has ended, which keeps the
 * two streams half a period apart (TSD_STAGGER=0 turns that off).  The kernel sequence of a batch runs eagerly the first time,
 * is captured into a CUDA graph the second time and replayed from then on (TSD_GRAPH=0: eager launches; none while profiling).
 * A batch's key includes its scratch slot, so a batch shape repeated in overlap mode runs eagerly on calls 1 and 2, is captured
 * on calls 3 and 4 and is replayed from call 5 on.  Up to 8 graphs are kept; a cycle of more than 8 keys runs eagerly.
 * tsd_stat_graphs counts captures and replays. */
TSD_API int tsd_flush(tsd_ctx *ctx);
/* Page-lock a caller-owned host buffer (cudaHostRegister, mapped).  tsd_detect_frames with TSD_MEM_HOST reads page-locked
 * frames IN PLACE over PCIe (only the 32-byte sectors the candidate ROIs touch are transferred, each once per batch, into a
 * device-resident mirror of the frames; batches of 512 frames or more run as up to four chunks whose transfers overlap the
 * previous chunk's kernels, TSD_STAGE_CHUNK=0 turns the chunking off); pageable frames are copied whole, in chunks that overlap
 * the kernels.  Buffers from cudaHostAlloc / torch pin_memory() are already page-locked.
 * Staging needs a 16-byte aligned frames pointer, row_stride and frame_stride multiples of 16 and 3 * W a multiple of 16; any other
 * page-locked layout is read by K2 itself, tap by tap over PCIe (as with TSD_STAGE=0).  Either way the records are the same. */
TSD_API int tsd_host_register(void *p, int64_t bytes);
TSD_API int tsd_host_unregister(void *p);
/* Number of kernels this library launched on the context since creation (bench.py's gpu_launches).  A replayed CUDA graph
 * counts the kernels it holds. */
TSD_API int64_t tsd_launch_count(tsd_ctx *ctx);
/* Measurement helper: CUDA graphs of the chain instantiated (*captured) and cached graphs launched again (*replayed) on the
 * context since its creation.  Host-side counters: does not synchronise. */
TSD_API int tsd_stat_graphs(tsd_ctx *ctx, int64_t *captured, int64_t *replayed);

/* ---- model / template state (host pointers) --------------------------------------------------------------- */
/* 6 red + 6 blue template masks, uint8 [6][D*D] in {0,255}: output of calculateMeanMasks (DET/source.py:24-59),
 * order = DET/constants.py SIGNALLIST.  Builds the bit-packed templates and the per-template score LUT
 * round(2TP/(TP+T), 2) (DET/source.py:563-567). */
TSD_API int tsd_set_templates(tsd_ctx *ctx, const uint8_t *red6, const uint8_t *blue6);
/* Optional override of the corner-similarity table f(d2) = EuclDSimilarity at squared distance d2 = 0..n-1
 * (DET/source.py:459-462).  By default the library fills it with libm pow(); the Python wrapper passes the
 * values numpy computes so that the in-process reference and the GPU path use bit-identical f.  TSD_E_INVALID unless
 * sqrt(f(n-1)) < coord_tol * merge_factor (pairs beyond the table take no action). */
TSD_API int tsd_set_similarity_table(tsd_ctx *ctx, const double *f, int n);
/* Six binary LDA classifiers: W f64 [nfeat][6] (column c = classifiers[c].coef_[0]), b f64 [6] (intercept_),
 * REC/source.py:551-562 fit on the host with scikit-learn.  nfeat = 1..4096 (324 for HOG, 1024 for raw grey pixels; the
 * chain needs 324).  K8 keeps W in shared memory, nfeat * 48 B: 192 KB at 4096 features; TSD_E_INVALID if the device
 * cannot give a block that much. */
TSD_API int tsd_set_lda(tsd_ctx *ctx, const double *W, const double *b, int nfeat);
/* 7-class LDA reducer + KNN training set: xbar f64 [nfeat], scalings f64 [nfeat][6], Ztrain f64 [ntrain][6],
 * ytrain int32 [ntrain] (REC/source.py:586-589).  k = 1..8, labels 0..15 (TSD_E_INVALID otherwise). */
TSD_API int tsd_set_knn(tsd_ctx *ctx, const double *xbar, const double *scalings, int nfeat, const double *Ztrain,
                        const int32_t *ytrain, int ntrain, int k);

/* ---- stage entry points ------------------------------------------------------------------------------------ */
/* K1  makeWindowBiggerOrDiscardFakeDetections (DET/source.py:155-174, REC/source.py:88-107), one result per box:
 * coords[i] (undefined when valid[i]==0), valid[i] in {0,1}. */
TSD_API int tsd_expand_boxes(tsd_ctx *ctx, const int32_t *boxes, int nboxes, double enlarge, int32_t *coords,
                             uint8_t *valid, int mem);

/* K2  cv2.resize(cropImageByCoords(coords, image), (D, D)) (DET/source.py:123-124,570-572; REC/source.py:57) for
 * n windows.  win_frame[i] = frame index of window i.  channels = 3 (BGR) or 1 (grey, REC/source.py:253-254). */
TSD_API int tsd_crop_resize(tsd_ctx *ctx, const uint8_t *frames, int nframes, int H, int W, int64_t row_stride,
                            int64_t frame_stride, int channels, const int32_t *coords, const int32_t *win_frame, int n,
                            int D, uint8_t *windows, int mem);

/* K1+K2 for whole frames: the candidate loop of MSERTrafficSignDetector (DET/source.py:116-124, REC/source.py:52-57).
 * Outputs are compacted per frame in MSER order: win_offsets [nframes+1], coords [cap][4], windows [cap][D][D][3],
 * cap >= box_offsets[nframes].  *total receives win_offsets[nframes]. */
TSD_API int tsd_windows(tsd_ctx *ctx, const uint8_t *frames, int nframes, int H, int W, int64_t row_stride,
                        int64_t frame_stride, const int32_t *boxes, const int32_t *box_offsets, double enlarge, int D,
                        uint8_t *windows, int32_t *coords, int32_t *win_offsets, int32_t *total, int mem);

/* K5  cleanDuplicatedDetections(list, by_coords, tol) per frame (DET/source.py:177-223; helpers :459-477,575-586).
 * In: windows/coords/offsets (CSR per frame).  Out: survivors, compacted per frame in the fold's list order.
 * *total_out receives out_offsets[nframes].  D = 2..32.  by_coords: TSD_E_INVALID unless tol * merge_factor (of the config) is
 * above sqrt(f(n-1)) of the similarity table, 0.3913 for the default one. */
TSD_API int tsd_dedup(tsd_ctx *ctx, const uint8_t *windows, const int32_t *coords, const int32_t *offsets, int nframes,
                      int D, int by_coords, double tol, uint8_t *out_windows, int32_t *out_coords, int32_t *out_offsets,
                      int32_t *total_out, int mem);

/* calculateHistAndNormalize (DET/source.py:575-586): float32 [n][50][60] min-max normalised H-S histograms. */
TSD_API int tsd_hist(tsd_ctx *ctx, const uint8_t *windows, int n, int D, float *hist, int mem);

/* Proposal pre-processing (SURVEY section 8(f) N1): grayAndEnhanceContrast (DET/source.py:135-152 = REC/source.py:67-84) for a
 * batch of frames: cv2.cvtColor(BGR2GRAY) -> cv2.createCLAHE(clipLimit, (tiles_x, tiles_y)).apply -> cv2.GaussianBlur((3,3), 0) ->
 * cv2.LUT(gamma table).  out uint8 [nframes][H][W] is what the reference hands to cv2.MSER.detectRegions (which stays on cv2).
 * The reference uses clip_limit = 2, tiles 8 x 8.  tsd_set_gamma_table replaces the default gammaCorrection(src, 2) table
 * (DET/source.py:599-605) with the caller's 256 bytes. */
TSD_API int tsd_set_gamma_table(tsd_ctx *ctx, const uint8_t *table256);
TSD_API int tsd_preprocess(tsd_ctx *ctx, const uint8_t *frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride,
                           double clip_limit, int tiles_x, int tiles_y, uint8_t *out, int mem);

/* Template builder (SURVEY section 8(f) N2): the running average of calculateMeanMasks (DET/source.py:44-52).  windows uint8
 * [n][D][D][3] (class crops already resized with tsd_crop_resize), group_offsets int32 [ngroups+1] (CSR, one group per sign
 * type, windows in the caller's os.listdir order -- the result depends on it): mean_out [ngroups][D][D][3] = first window,
 * then cv2.addWeighted(window, .5, mean, .5, 0) for every further one.  Host pointers only. */
TSD_API int tsd_mean_windows(tsd_ctx *ctx, const uint8_t *windows, const int32_t *group_offsets, int ngroups, int D,
                             uint8_t *mean_out, int mem);

/* N4 (reporting)  The matching loops of the evaluators.  Host pointers.
 * tsd_match_detections = checkIfDetectionByTypeOnFileIsCorrectIncorrectDuplicated + getCorrectsAndWrongByTypeOnFile
 * (DET/source.py:401-450) for all files and types at once: det / gt int32 [n][6] = (frame, x1, y1, x2, y2, type bucket 0..5), gt grouped
 * by frame (gt_offsets int32 [nframes+1]); status int32 [ndet] (1 = "correct": best same-type ground truth by
 * sqrt(f(d_TL) f(d_BR)) exceeds tol = 0.85), match int32 [ndet] (its gt row or -1), tally int32 [nframes][6][4] =
 * (correct, incorrect, not detected, expected).  Needs tsd_set_similarity_table.  TSD_E_INVALID unless tol is above sqrt(f(n-1)) of
 * the table (0.3913 for 65 536 entries): ground truths beyond the table are skipped. */
TSD_API int tsd_match_detections(tsd_ctx *ctx, const int32_t *det, int ndet, const int32_t *gt, const int32_t *gt_offsets, int nframes,
                                 double tol, int32_t *status, int32_t *match, int32_t *tally);
/* tsd_match_iou = the loop of precision_recall_curve (Reconocimiento de Objetos/evaluar_resultados.py:224-262) with bboxes_overlap
 * (:53-89): det int32 [ndet][5] = (left, top, right, bottom, index in the score-descending list) grouped by image and, inside an
 * image, in list order (det_offsets int32 [nimages+1]); gt int32 [ngt][5] = (left, top, right, bottom, class; -1 = ignore region)
 * grouped by image (gt_offsets); tp / fp uint8 [ndet] indexed by list position. */
TSD_API int tsd_match_iou(tsd_ctx *ctx, const int32_t *det, const int32_t *det_offsets, const int32_t *gt, const int32_t *gt_offsets,
                          int nimages, double ovr, uint8_t *tp, uint8_t *fp);

/* K3  getColorMaskRedOrBlue(img, 'r') and (img, 'b') (DET/source.py:63-89): uint8 [n][D*D] in {0,255} each. */
TSD_API int tsd_color_masks(tsd_ctx *ctx, const uint8_t *windows, int n, int D, uint8_t *red, uint8_t *blue, int mem);
/* cv2.cvtColor(BGR2HSV) (DET/source.py:65,576) for npx pixels. */
TSD_API int tsd_bgr2hsv(tsd_ctx *ctx, const uint8_t *bgr, int64_t npx, uint8_t *hsv, int mem);

/* K4  getSimilarSignalType x2 + the decision of detectionsMaskCorrelation (DET/source.py:229-261,545-567).
 * scores int32 [n][2][6] = hundredths of calculateScoreBetweenMatrixs per (red|blue, template) (may be NULL);
 * id int32 [n] (1..6), hundredths int32 [n] (winner's score), emit uint8 [n] (winner > tol). */
TSD_API int tsd_score_masks(tsd_ctx *ctx, const uint8_t *red, const uint8_t *blue, int n, int D, int32_t *scores,
                            int32_t *id, int32_t *hundredths, uint8_t *emit, int mem);

/* K3 + K4 in one call: detectionsMaskCorrelation (DET/source.py:229-245) for n windows uint8 [n][D][D][3] -> id (1..6), hundredths of
 * the winner's score, emit (winner > tolerance).  Host pointers. */
TSD_API int tsd_score(tsd_ctx *ctx, const uint8_t *windows, int n, int D, int32_t *id, int32_t *hundredths, uint8_t *emit, int mem);

/* K6  cv2.cvtColor(BGR2GRAY) (REC/source.py:388): uint8 [npx]. */
TSD_API int tsd_bgr2gray(tsd_ctx *ctx, const uint8_t *bgr, int64_t npx, uint8_t *gray, int mem);
/* K7  computeDescriptors(img, (hog,'HOG')) = cv2.HOGDescriptor.compute (REC/source.py:517-521,487-494):
 * gray uint8 [n][32][32] -> float32 [n][324]. */
TSD_API int tsd_hog(tsd_ctx *ctx, const uint8_t *gray, int n, float *desc, int mem);
/* K8  predictProbabilityLDAClassifiers + extractBestPredictions (REC/source.py:565-577,627-641,342-347):
 * X float32 [n][nfeat] -> logits f64 [n][6] (may be NULL), labels int32 [n] (0 = no sign). */
TSD_API int tsd_lda_predict(tsd_ctx *ctx, const float *X, int n, double tol, double *logits, int32_t *labels, int mem);
/* K6 + K7 + K8 in one call for n BGR windows uint8 [n][32][32][3]: BGR2GRAY (REC/source.py:388), HOG (:519), predict_proba x6 and
 * extractBestPredictions (:565-577,627-641) -> labels int32 [n] (0 = no sign).  Host pointers. */
TSD_API int tsd_recognize(tsd_ctx *ctx, const uint8_t *windows, int n, double tol, int32_t *labels, int mem);

/* EVALUATION ONLY (BASELINE.json north_star: the LDA projection on tensor cores vs FMA): the same decision from mma.sync TF32 logits,
 * split = 1 (plain TF32) or 3 (3xTF32 with FP32 accumulation).  logits float32 [n][6] (may be NULL), *ms (may be NULL) = device time of
 * the kernel alone.  The chain and tsd_lda_predict use the f64 FMA kernel (the reference computes in float64).  Host pointers.
 * The kernel keeps W as TF32 tiles in shared memory, 64 B per feature rounded up to 8 features: TSD_E_INVALID when they do not fit
 * in one block (above 3 632 features on the B200). */
TSD_API int tsd_lda_predict_tf32(tsd_ctx *ctx, const float *X, int n, double tol, int split, float *logits, int32_t *labels, float *ms, int mem);

/* K8b predictProbabilityKNNClassifiers (REC/source.py:592-596): Z f64 [n][6] (may be NULL), labels int32 [n].
 * Brute force over the training set; training rows at equal distance are ranked by index (the smaller one is nearer), then a
 * uniform vote with ties to the smallest label.  scikit-learn's kd-tree orders exact distance ties its own way, so labels can
 * differ from it when a tie straddles the k-th neighbour (SURVEY A.8). */
TSD_API int tsd_knn_predict(tsd_ctx *ctx, const float *X, int n, double *Z, int32_t *labels, int mem);

/* ---- whole path -------------------------------------------------------------------------------------------- */
/* One detection record = one line of resultado.txt (DET/source.py:501-508). */
typedef struct tsd_detection {
    int32_t frame;             /* index into the batch */
    int32_t x1, y1, x2, y2;    /* as reported by the reference: x2,y2 are NOT clipped to the frame */
    int32_t id;                /* 1..6 (detection) ; 0..6 label (recognition) */
    int32_t hundredths;        /* score * 100 (detection) ; 0 for recognition */
    int32_t reserved;
} tsd_detection;

#define TSD_RUN_DETECT 1       /* K1 K2 K5 K5 K3 K4  (DET main.py path) */
#define TSD_RUN_RECOGNIZE 2    /* K1 K2 K5 K5 K6 K7 K8 on the recognition flavour (x1.15, 32x32) */

/* The whole post-MSER chain for a batch of frames (SURVEY.md section 3.4):
 * MSERTrafficSignDetector's candidate loop + both cleanDuplicatedDetections passes (DET/source.py:116-131), then
 * detectionsMaskCorrelation for every survivor (DET/source.py:708-716)  [TSD_RUN_DETECT], or
 * BGR2GRAY + HOG + LDA decision [TSD_RUN_RECOGNIZE].
 * det [det_cap] receives the records in frame order then list order; counts int32 [4] (may be NULL) receives
 * {raw boxes, aspect-passing windows, survivors, detections}.  Returns TSD_E_NOMEM if det_cap is too small.
 * With TSD_MEM_DEVICE the frames/boxes are device memory, `det`/`counts` are still HOST pointers and the call
 * synchronises once at the end. */
TSD_API int tsd_detect_frames(tsd_ctx *ctx, int mode, const uint8_t *frames, int nframes, int H, int W,
                              int64_t row_stride, int64_t frame_stride, const int32_t *boxes,
                              const int32_t *box_offsets, tsd_detection *det, int det_cap, int32_t *ndet,
                              int32_t *counts, int mem);

/* Same chain, device-resident and asynchronous: enqueues the kernels on the context's stream and returns.  Results
 * stay in context-owned device buffers; fetch them with tsd_fetch_detections (which synchronises).  bench.py times
 * this call with CUDA events.  max_boxes_per_frame = largest box_offsets[f+1]-box_offsets[f] (sizes the per-frame
 * pair matrix of K5); pass 0 to let the library read the offsets back (one small synchronising copy). */
TSD_API int tsd_enqueue_frames(tsd_ctx *ctx, int mode, const uint8_t *d_frames, int nframes, int H, int W,
                               int64_t row_stride, int64_t frame_stride, const int32_t *d_boxes,
                               const int32_t *d_box_offsets, int nboxes_total, int max_boxes_per_frame);
TSD_API int tsd_fetch_detections(tsd_ctx *ctx, tsd_detection *det, int det_cap, int32_t *ndet, int32_t *counts);
/* Streaming use of the two slots: after  enqueue(batch k); enqueue(batch k+1);  tsd_fetch_previous returns batch k's records
 * (same arguments as tsd_fetch_detections) while batch k+1 keeps running -- e.g. its K2 pulling ROIs out of page-locked host
 * frames over PCIe under batch k's GPU-bound kernels.  TSD_E_STATE if there is no such batch. */
TSD_API int tsd_fetch_previous(tsd_ctx *ctx, tsd_detection *det, int det_cap, int32_t *ndet, int32_t *counts /* [4] or NULL */);

/* Measurement helper: total number of non-zero histogram bins over the windows of the last tsd_enqueue_frames call, each
 * window as the first duplicate-removal pass leaves it: an item that absorbed a near duplicate counts the histogram of its
 * merged pixels (the fold rebuilds it in place).  It approximates the bytes k5_pairs has to read at least once.  Synchronises. */
TSD_API int tsd_stat_hist_entries(tsd_ctx *ctx, int64_t *total);

/* Measurement helper: number of window pairs (since process start, this device) whose class could not be decided from the exact
 * integer dot product -- cv2.compareHist's value within 2e-6 of a threshold of DET/source.py:203-217 -- and was therefore computed
 * with the exact float64 evaluation.  reset != 0 zeroes the counter.  Synchronises. */
TSD_API int tsd_stat_unsure_pairs(tsd_ctx *ctx, int64_t *total, int reset);

/* Measurement helper: bytes that crossed PCIe host -> device for the frames of tsd_detect_frames calls on page-locked host memory
 * (every 32-byte sector the candidate ROIs of a batch touch is copied once), since process start / the last reset.  Synchronises. */
TSD_API int tsd_stat_staged_bytes(tsd_ctx *ctx, int64_t *total, int reset);

/* Device-side stage timing: CUDA events are recorded between the stages of every tsd_enqueue_frames call made after
 * tsd_set_profiling(ctx, 1); tsd_stage_times synchronises and returns, per stage name, the time summed over those
 * calls (names[i] / ms[i] for i < returned count). */
TSD_API int tsd_set_profiling(tsd_ctx *ctx, int on);
TSD_API int tsd_stage_times(tsd_ctx *ctx, const char **names, float *ms, int cap);
/* tsd_set_profiling(ctx, 2) keeps consecutive tsd_enqueue_frames calls overlapped (two scratch slots, two streams) and
 * tsd_timeline returns every stage boundary recorded since then, in enqueue order, as milliseconds after the first one
 * (names[i] stay valid until the next call on the context).  Synchronises. */
TSD_API int tsd_timeline(tsd_ctx *ctx, const char **names, float *ms, int cap);

#ifdef __cplusplus
}
#endif
#endif /* TSD_B200_H */
