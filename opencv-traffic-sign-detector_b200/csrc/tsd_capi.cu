// tsd_capi.cu -- C-ABI shared library (include/tsd_b200.h) over the sm_100a kernels in tsd_kernels.cuh.
// Host side: context, grow-only device scratch, stream-ordered staging for host-pointer calls, the batched chain.
// There is no CPU fallback anywhere in this file: every entry point launches CUDA kernels or fails.
#include "../../include/tsd_b200.h"
#include "tsd_kernels.cuh"
#include "tsd_k5.cuh"
#include "tsd_k2_tma.cuh"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

using namespace tsd;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                             \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess) return fail(TSD_E_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)
#define TRY(call)                 \
    do {                          \
        int r_ = (call);          \
        if (r_ != TSD_OK) return r_; \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct tsd_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t cur = nullptr;              // the stream kernels are launched on (== stream except inside an overlapped enqueue)
    // One batch = one tsd_enqueue_frames call.  wo / fo = first window slot / first per-frame entry of the batch in the scratch arrays,
    // nbcap = upper bound of its windows, sidx = its record in b_summary.
    struct Batch { int nframes = 0; size_t wo = 0; int fo = 0; int nbcap = 0; int sidx = 0; int nboxes = 0; bool valid = false, in_slot = false; };
    Batch last, prev;                        // the last enqueue / the one before it (overlap mode: tsd_fetch_previous)
    // Default (TSD_OVERLAP=0 turns it off): consecutive tsd_enqueue_frames calls alternate between two scratch slots and two streams, so the latency-bound
    // fold of one batch runs under the throughput-bound kernels of the next.  tsd_stream() is ordered after a batch only once the
    // NEXT call, tsd_flush, tsd_synchronize or tsd_fetch_detections has been issued (the join is deferred by one call).
    int overlap = 1, slot = 0, pending_join = -1;
    size_t slot_cap = 0, slot_fcap = 0, slot_todo = 0;   // windows / per-frame entries / k5_pairs work-list entries per slot
    int slot_rw = 1;                         // words per bit row of the pair-class matrix the slot layout is sized for (sticky maximum)
    cudaEvent_t ev_slot_fork[2] = {nullptr, nullptr}, ev_join[2] = {nullptr, nullptr};
    cudaEvent_t ev_w1[2] = {nullptr, nullptr};   // slot's batch has finished its throughput-bound front half (K1 .. pair classes)
    int stagger = 1;                         // TSD_STAGGER: the front half of a batch starts only when the previous batch's has ended
    cudaStream_t os[2] = {nullptr, nullptr};                                // per slot: the chain's stream
    DevBuf b_summary, b_order, b_gramdone;
    unsigned* d_tickets = nullptr;           // zero-initialised counters of the last-CTA-done scans: [slot 0 | slot 1 | stage calls] x 8
    int ticket_base = 16;
    size_t order_off = 0;                    // offset (ints) of the current batch inside b_order
    cudaStream_t copy_stream = nullptr;      // host-buffer calls: H2D of the next chunk of frames overlaps the chain on `stream`
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
    DevBuf b_stage[2], b_hboxes, b_hoff;
    int zero_copy = 1;                       // page-locked host frames are read in place over PCIe (TSD_ZEROCOPY=0: always copy whole frames)
    int stage_rois = 1;                      // ... by the mark + copy kernels, each touched 32-byte sector once, into a device mirror K2 reads
                                             // (TSD_STAGE=0: K2 itself gathers from host memory, round 1's path)
    DevBuf b_mirror[2], b_stagemap[2];       // per scratch slot (consecutive batches of a chunked tsd_detect_frames call overlap)
    int stage_chunk = 256;                   // TSD_STAGE_CHUNK: frames per chunk of tsd_detect_frames on page-locked host frames (0 = one batch)
    int stage_ctas = 2;                      // TSD_STAGE_CTAS: CTAs per SM of the staging copy (PCIe-bound: 2 keep the link as busy as 8 and leave the SMs to the other chunk's chain)
    int stage_gran = 1;                      // TSD_STAGE_GRAN = 32 | 64 | 128 bytes: unit the marked spans are widened to (sectors: 1, 2, 4)
    unsigned long long* d_staged = nullptr;  // bytes the staging copy moved over PCIe (tsd_stat_staged_bytes)
    int chunk_frames = 32;                   // TSD_CHUNK_FRAMES: frames per H2D chunk of the host-buffer path
    tsd_config cfg;
    int64_t launches = 0;
    int sm_count = 148;
    // constant state
    Tables* d_tab = nullptr;
    ScoreTemplates* d_tmpl = nullptr;
    uint8_t* d_gamma = nullptr;              // gammaCorrection table (DET:599-605), 256 bytes
    DevBuf b_pgray, b_pluts, b_pin, b_pout;  // pre-processing scratch
    MaskLut* d_mlut = nullptr;               // inRange bounds of tsd_config as per-channel flag tables (K3)
    bool have_templates = false;
    int tmpl_D = 0;
    double* d_simtab = nullptr;
    int simtab_n = 0;
    std::vector<double> h_simtab;
    double* d_ldaW = nullptr; double* d_ldab = nullptr; int lda_nfeat = 0;
    double* d_xbar = nullptr; double* d_scal = nullptr; double* d_Zt = nullptr; int32_t* d_yt = nullptr;
    int knn_nfeat = 0, knn_ntrain = 0, knn_k = 4;
    HogConst hog;
    // grow-only scratch
    DevBuf b_coords, b_winframe, b_windows, b_entries, b_meta, b_list, b_flags, b_cnt, b_winoff, b_survcnt, b_survoff,
        b_slots, b_pairs, b_energy, b_red, b_blue, b_bits, b_id, b_hund, b_emit, b_detcnt, b_detoff, b_det, b_gray, b_hog, b_labels, b_scores;
    int last_mode = 0;
    int profiling = 0;
    int keep_masks = 0;                      // TSD_KEEP_MASKS=1: the chain also writes K3's byte masks (nobody reads them there)
    int use_gram = 1;                        // TSD_GRAM=0: pair classes of every frame from the CUDA-core kernel (k5_pairs)
    int k2_grid = 256;                       // TSD_K2_GRID: CTAs per SM of K2 (0 = one window per warp, no loop).  4096 frames, ms: 12: .830, 24: .784, 48: .741, 96: .718, 128: .715, 192: .708, 256: .709, 384: .704, 640: .709, unlimited (1384): .757
    int fold_per_sm_cap = 2;                 // TSD_FOLD_PER_SM: cap of resident k5_fold_warp CTAs per SM (0 = as many as fit; measured with the staggered overlap at 4096 frames: 0: 3.22, 1: 3.20, 2: 3.09, 3: 3.18 ms per step)
    int fold_cta_cost = 0;                   // TSD_FOLD_CTA_COST: frames with at least this many merge-band pairs go to the CTA fold (0 = by size only)
    // function attributes (dynamic shared memory opt-in) are set once per context: per-context flags, no process-wide statics
    int fold_per_sm[4] = {0, 0, 0, 0};       // resident CTAs per SM of the four k5_fold_warp instantiations (0 = not queried yet)
    bool attr_gram = false, attr_pairs = false, attr_k2tma = false;
    int k2_tma = 0;                          // TSD_K2=tma: the TMA-staged resize kernel (tsd_k2_tma.cuh) instead of the direct gather
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> ev_names;
    int ev_used = 0;
    // CUDA graphs of the chain (TSD_GRAPH=0 turns them off): a batch shape seen twice in a row is captured once and replayed from then
    // on -- the chains of small batches (real MSER frames) are bound by launch latency.  `gen` counts every event that changes a
    // pointer baked into a captured kernel argument (scratch reallocation, slot layout, model state) and is part of the key.
    struct GraphEntry { std::vector<uint64_t> key; cudaGraphExec_t exec = nullptr; int64_t launches = 0; uint64_t stamp = 0; };
    std::vector<GraphEntry> graphs;
    std::vector<uint64_t> seen_key;
    uint64_t gen = 0, graph_clock = 0;
    int use_graph = 1;
};

static int ensure(tsd_ctx* c, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return TSD_OK;
    if (b.p) { CU(cudaStreamSynchronize(c->stream)); CU(cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
    c->gen++;                                                // captured graphs hold the old pointer
    size_t want = bytes + bytes / 4 + 256;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return TSD_OK;
}

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

static int check_launch(tsd_ctx* c, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(TSD_E_CUDA, "launch %s: %s", what, cudaGetErrorString(e));
    c->launches++;
    return TSD_OK;
}

// Lets kernel fn launch with `bytes` of dynamic shared memory: fails with TSD_E_INVALID when the device's per-block opt-in limit
// is smaller (227 KB on the B200), else raises the function's limit.  Never lowers it: the attribute belongs to the device, and
// another context on it may need a larger value.
static int allow_dynamic_smem(tsd_ctx* c, const void* fn, size_t bytes, const char* what) {
    int optin = 0;
    CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, fn));
    if (bytes + fa.sharedSizeBytes > (size_t)optin)
        return fail(TSD_E_INVALID, "%s needs %zu B of shared memory per block, the device allows %d B", what, bytes + fa.sharedSizeBytes, optin);
    if (bytes > (size_t)fa.maxDynamicSharedSizeBytes) CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return TSD_OK;
}

// Event record / wait on c->cur that also works while the stream is being captured into a CUDA graph (external event nodes).
static int ev_record(tsd_ctx* c, cudaEvent_t ev) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    CU(cudaStreamIsCapturing(c->cur, &st));
    CU(cudaEventRecordWithFlags(ev, c->cur, st == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
    return TSD_OK;
}
static int ev_wait(tsd_ctx* c, cudaEvent_t ev) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    CU(cudaStreamIsCapturing(c->cur, &st));
    CU(cudaStreamWaitEvent(c->cur, ev, st == cudaStreamCaptureStatusActive ? cudaEventWaitExternal : cudaEventWaitDefault));
    return TSD_OK;
}

static void mark(tsd_ctx* c, const char* name) {
    if (!c->profiling) return;
    if (c->ev_used >= (int)c->ev.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        c->ev.push_back(e);
        c->ev_names.push_back("");
    }
    c->ev_names[c->ev_used] = name;
    cudaEventRecord(c->ev[c->ev_used], c->cur);
    c->ev_used++;
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" {

const char* tsd_last_error(void) { return g_err; }
const char* tsd_version(void) { return "tsd_b200 0.1 (sm_100a)"; }

int tsd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int tsd_config_default(tsd_config* cfg, int flavour) {
    if (!cfg) return fail(TSD_E_INVALID, "cfg is NULL");
    memset(cfg, 0, sizeof *cfg);
    cfg->enlarge = flavour == 1 ? 1.15 : 1.30;
    cfg->aspect_lo = 0.8; cfg->aspect_hi = 1.20;
    cfg->window = flavour == 1 ? 32 : 25;
    cfg->score_tol_hundredths = 55;
    cfg->hist_tol = 0.85; cfg->coord_tol = 0.95; cfg->merge_factor = 0.8823;
    const uint8_t rl[2][3] = {{0, 50, 10}, {160, 50, 10}}, rh[2][3] = {{10, 255, 255}, {179, 255, 255}};
    memcpy(cfg->red_lo, rl, 6); memcpy(cfg->red_hi, rh, 6);
    const uint8_t bl[3] = {90, 70, 10}, bh[3] = {128, 255, 255};
    memcpy(cfg->blue_lo, bl, 3); memcpy(cfg->blue_hi, bh, 3);
    cfg->proba_tol = 0.5; cfg->knn_k = 4;
    return TSD_OK;
}

static double eucl_similarity_d2(long long d2) {             // DET:459-462 with libm
    if (d2 <= 0) return 1.0;
    double d = sqrt((double)d2);
    return 1.0 / (1.0 + pow(M_E, ((0.154 * pow(d, 1.2)) - 31.8) / (0.2 * d)));
}

// Pairs whose squared corner distance is at or beyond the similarity table take no action (coord_sim, eval_match).  That equals
// the reference only while every such pair's similarity stays below the lowest one that acts, `lo`: f is decreasing, so the table
// must reach a distance where sqrt(f(n-1)) < lo.  (The default table reaches 255 px: sqrt(f(65535)) = 0.3913.)
static int check_simtab(const tsd_ctx* c, double lo, const char* what) {
    const double s = sqrt(c->h_simtab[c->simtab_n - 1]);
    if (s >= lo) return fail(TSD_E_INVALID, "%s %.6g is not above sqrt(f(%d)) = %.6g: the corner-similarity table is too short", what, lo, c->simtab_n - 1, s);
    return TSD_OK;
}

static int create_impl(tsd_ctx* c, int device) {
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    c->cur = c->stream;
    for (int i = 0; i < 2; i++) {
        CU(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
        CU(cudaStreamCreateWithFlags(&c->os[i], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&c->ev_slot_fork[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_w1[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_consumed[i], cudaEventDisableTiming));
    }
    { const char* e = getenv("TSD_OVERLAP"); if (e) c->overlap = atoi(e) != 0; }
    { const char* e = getenv("TSD_ZEROCOPY"); if (e) c->zero_copy = e[0] != '0'; }
    { const char* e = getenv("TSD_STAGE"); if (e) c->stage_rois = e[0] != '0'; }
    { const char* e = getenv("TSD_STAGE_GRAN"); if (e) { const int g = atoi(e); c->stage_gran = g >= 128 ? 4 : g >= 64 ? 2 : 1; } }
    { const char* e = getenv("TSD_CHUNK_FRAMES"); if (e && atoi(e) > 0) c->chunk_frames = atoi(e); }
    { const char* e = getenv("TSD_STAGE_CHUNK"); if (e) c->stage_chunk = atoi(e); }
    { const char* e = getenv("TSD_STAGE_CTAS"); if (e && atoi(e) > 0) c->stage_ctas = atoi(e); }
    { const char* e = getenv("TSD_KEEP_MASKS"); if (e) c->keep_masks = atoi(e); }
    { const char* e = getenv("TSD_GRAM"); if (e) c->use_gram = atoi(e) != 0; }
    { const char* e = getenv("TSD_GRAPH"); if (e) c->use_graph = atoi(e) != 0; }
    { const char* e = getenv("TSD_K2"); if (e) c->k2_tma = strcmp(e, "tma") == 0; }
    { const char* e = getenv("TSD_FOLD_CTA_COST"); if (e) c->fold_cta_cost = atoi(e); }
    { const char* e = getenv("TSD_FOLD_PER_SM"); if (e) c->fold_per_sm_cap = atoi(e); }
    { const char* e = getenv("TSD_STAGGER"); if (e) c->stagger = atoi(e); }
    { const char* e = getenv("TSD_K2_GRID"); if (e) c->k2_grid = atoi(e); }
    {   // keep stream-ordered temporaries cached in the pool instead of returning them to the OS at every synchronise
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    // tables (SURVEY A.3 / A.5)
    Tables t;
    t.sdiv[0] = t.hdiv[0] = 0;
    for (int i = 1; i < 256; i++) {
        t.sdiv[i] = (int32_t)lrint((255 << 12) / (1. * i));
        t.hdiv[i] = (int32_t)lrint((180 << 12) / (6. * i));
    }
    const double a_h = 50 / (180. - 0.), a_s = 60 / (256. - 0.);
    for (int i = 0; i < 256; i++) {
        int hb = (int)floor(i * a_h + (-0. * a_h)), sb = (int)floor(i * a_s + (-0. * a_s));
        t.hbin[i] = (uint8_t)(hb < kHistH ? hb : kHistH - 1);
        t.sbin[i] = (uint8_t)(sb < kHistS ? sb : kHistS - 1);
        // the histogram kernels compute both bins arithmetically (hue_bin, (S * 60) >> 8): they must agree with calcHist's float rule
        if ((i < 180 && hue_bin(i) != t.hbin[i]) || ((i * kHistS) >> 8) != t.sbin[i]) return fail(TSD_E_STATE, "histogram bin arithmetic disagrees with the table at %d", i);
    }
    CU(cudaMalloc(&c->d_tab, sizeof(Tables)));
    CU(cudaMemcpy(c->d_tab, &t, sizeof t, cudaMemcpyHostToDevice));
    CU(cudaMalloc(&c->d_tmpl, sizeof(ScoreTemplates)));
    CU(cudaMalloc(&c->d_tickets, 24 * sizeof(unsigned)));
    CU(cudaMalloc(&c->d_staged, 8));
    CU(cudaMemset(c->d_staged, 0, 8));
    CU(cudaMemset(c->d_tickets, 0, 24 * sizeof(unsigned)));
    {   // default gamma table: ((i / 255) ** (1 / 2)) * 255 truncated to uint8 (DET:602-603); the Python wrapper overrides it with the
        // table the reference's own expression gives in-process
        uint8_t gt[256];
        for (int i = 0; i < 256; i++) gt[i] = (uint8_t)(pow(i / 255.0, 1.0 / 2.0) * 255.0);
        CU(cudaMalloc(&c->d_gamma, 256));
        CU(cudaMemcpy(c->d_gamma, gt, 256, cudaMemcpyHostToDevice));
    }
    {   // K3 flag tables: bit 0 / 1 = red band 0 / 1, bit 2 = blue (DET:70-86 bounds from the config)
        MaskLut ml;
        const tsd_config& g = c->cfg;
        for (int v = 0; v < 256; v++) {
            uint8_t f[3] = {0, 0, 0};
            for (int ch3 = 0; ch3 < 3; ch3++) {
                if (v >= g.red_lo[0][ch3] && v <= g.red_hi[0][ch3]) f[ch3] |= 1;
                if (v >= g.red_lo[1][ch3] && v <= g.red_hi[1][ch3]) f[ch3] |= 2;
                if (v >= g.blue_lo[ch3] && v <= g.blue_hi[ch3]) f[ch3] |= 4;
            }
            ml.hf[v] = f[0]; ml.sf[v] = f[1]; ml.vf[v] = f[2];
        }
        CU(cudaMalloc(&c->d_mlut, sizeof(MaskLut)));
        CU(cudaMemcpy(c->d_mlut, &ml, sizeof ml, cudaMemcpyHostToDevice));
    }
    // default corner-similarity table
    const int n = 1 << 16;
    std::vector<double> f(n);
    for (int i = 0; i < n; i++) f[i] = eucl_similarity_d2(i);
    CU(cudaMalloc(&c->d_simtab, sizeof(double) * n));
    CU(cudaMemcpy(c->d_simtab, f.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
    c->simtab_n = n;
    c->h_simtab = f;
    TRY(check_simtab(c, c->cfg.coord_tol * c->cfg.merge_factor, "coord_tol * merge_factor ="));
    {   // HOG Gaussian window, sigma = (16+16)/8 = 4  (OpenCV HOGCache::init)
        float sigma = 4.f, sc = 1.f / (sigma * sigma * 2);
        for (int i = 0; i < 16; i++) {
            const float di = i - 16 * 0.5f, g = expf(-di * di * sc);
            const float cell = (i + 0.5f) / 8 - 0.5f;
            const int i0 = (int)floorf(cell);
            const float f = cell - i0;
            for (int cc = 0; cc < 2; cc++) {
                float wgt = 0.f;                             // bilinear weight of cell cc at position i (out-of-range neighbours dropped)
                if (cc == i0) wgt = 1.f - f; else if (cc == i0 + 1) wgt = f;
                c->hog.wsep[i][cc] = g * wgt;
            }
        }
    }
    return TSD_OK;
}

int tsd_create(tsd_ctx** out, int device, const tsd_config* cfg) {
    if (!out) return fail(TSD_E_INVALID, "ctx out pointer is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(TSD_E_CUDA, "no CUDA device available (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
    if (device < 0 || device >= ndev) return fail(TSD_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
    CU(cudaSetDevice(device));
    tsd_ctx* c = new tsd_ctx();
    c->device = device;
    if (cfg) c->cfg = *cfg; else tsd_config_default(&c->cfg, 0);
    if (c->cfg.window < 2 || c->cfg.window > kMaxD) { delete c; return fail(TSD_E_INVALID, "window %d not in [2,%d]", c->cfg.window, kMaxD); }
    const int rc = create_impl(c, device);
    if (rc != TSD_OK) { tsd_destroy(c); return rc; }         // one cleanup path: whatever was created so far is released (g_err is kept)
    *out = c;
    return TSD_OK;
}

int tsd_destroy(tsd_ctx* c) {
    if (!c) return TSD_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (int i = 0; i < 2; i++) if (c->os[i]) cudaStreamSynchronize(c->os[i]);
    DevBuf* bufs[] = {&c->b_coords, &c->b_winframe, &c->b_windows, &c->b_entries, &c->b_meta, &c->b_list, &c->b_flags, &c->b_cnt,
                      &c->b_winoff, &c->b_survcnt, &c->b_survoff, &c->b_slots, &c->b_pairs, &c->b_energy, &c->b_red, &c->b_blue, &c->b_bits, &c->b_id, &c->b_hund,
                      &c->b_emit, &c->b_detcnt, &c->b_detoff, &c->b_det, &c->b_gray, &c->b_hog, &c->b_labels, &c->b_scores,
                      &c->b_stage[0], &c->b_stage[1], &c->b_hboxes, &c->b_hoff, &c->b_summary, &c->b_order, &c->b_gramdone, &c->b_mirror[0], &c->b_mirror[1], &c->b_stagemap[0], &c->b_stagemap[1], &c->b_pgray, &c->b_pluts, &c->b_pin, &c->b_pout};
    for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
    for (int i = 0; i < 2; i++) {
        if (c->ev_slot_fork[i]) cudaEventDestroy(c->ev_slot_fork[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
        if (c->ev_w1[i]) cudaEventDestroy(c->ev_w1[i]);
        if (c->os[i]) cudaStreamDestroy(c->os[i]);
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
        if (c->ev_consumed[i]) cudaEventDestroy(c->ev_consumed[i]);
    }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    void* ptrs[] = {c->d_staged, c->d_tickets, c->d_tab, c->d_tmpl, c->d_mlut, c->d_gamma, c->d_simtab, c->d_ldaW, c->d_ldab, c->d_xbar, c->d_scal, c->d_Zt, c->d_yt};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
    for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return TSD_OK;
}

void* tsd_stream(tsd_ctx* c) { return c ? (void*)c->stream : nullptr; }

int tsd_host_register(void* p, int64_t bytes) {
    if (!p || bytes <= 0) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaHostRegister(p, (size_t)bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return TSD_OK;
}

int tsd_host_unregister(void* p) {
    if (!p) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaHostUnregister(p));
    return TSD_OK;
}

// TSD_OVERLAP: make the context's stream wait for the batch enqueued last (its join was deferred)
static int join_pending(tsd_ctx* c) {
    if (c->pending_join >= 0) { CU(cudaStreamWaitEvent(c->stream, c->ev_join[c->pending_join], 0)); c->pending_join = -1; }
    return TSD_OK;
}

int tsd_flush(tsd_ctx* c) {
    if (!c) return fail(TSD_E_INVALID, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    return join_pending(c);
}

int tsd_synchronize(tsd_ctx* c) {
    if (!c) return fail(TSD_E_INVALID, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int64_t tsd_launch_count(tsd_ctx* c) { return c ? c->launches : 0; }

int tsd_set_profiling(tsd_ctx* c, int on) {
    if (!c) return fail(TSD_E_INVALID, "ctx is NULL");
    TRY(join_pending(c));
    c->profiling = on;                                       // 1: per-stage times, batches serialised; 2: timeline, batches overlapped as usual (both without CUDA graphs)
    c->ev_used = 0;                                          // (re)start accumulating
    return TSD_OK;
}

// Sums, per stage name, the CUDA-event time between consecutive marks of every tsd_enqueue_frames call made since
// tsd_set_profiling(ctx, 1).  Synchronises the stream.
int tsd_stage_times(tsd_ctx* c, const char** names, float* ms, int cap) {
    if (!c) return fail(TSD_E_INVALID, "ctx is NULL");
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    static thread_local std::vector<std::string> uniq;
    uniq.clear();
    std::vector<float> sum;
    for (int i = 1; i < c->ev_used; i++) {
        if (c->ev_names[i] == "start") continue;
        float t = 0;
        cudaEventElapsedTime(&t, c->ev[i - 1], c->ev[i]);
        size_t k = 0;
        while (k < uniq.size() && uniq[k] != c->ev_names[i]) k++;
        if (k == uniq.size()) { uniq.push_back(c->ev_names[i]); sum.push_back(0.f); }
        sum[k] += t;
    }
    int n = 0;
    for (size_t k = 0; k < uniq.size() && n < cap; k++, n++) { names[n] = uniq[k].c_str(); ms[n] = sum[k]; }
    return n;
}

// tsd_set_profiling(ctx, 2): every mark since then as (name, milliseconds after the first mark), in enqueue order -- the batches
// keep overlapping, so this is the timeline of the two-slot pipeline.  Synchronises.
int tsd_timeline(tsd_ctx* c, const char** names, float* ms, int cap) {
    if (!c) return fail(TSD_E_INVALID, "ctx is NULL");
    cudaSetDevice(c->device);
    TRY(join_pending(c));
    cudaStreamSynchronize(c->stream);
    int n = 0;
    for (int i = 0; i < c->ev_used && n < cap; i++, n++) {
        float t = 0;
        if (i) cudaEventElapsedTime(&t, c->ev[0], c->ev[i]);
        names[n] = c->ev_names[i].c_str();
        ms[n] = t;
    }
    return n;
}

// ---- state ------------------------------------------------------------------------------------------------------
static int round2_hundredths(double v) {                     // Python round(v, 2): exactly rounded decimal (DET:567)
    char buf[64];
    snprintf(buf, sizeof buf, "%.2f", v);
    return (int)lrint(strtod(buf, NULL) * 100.0);
}

int tsd_set_templates(tsd_ctx* c, const uint8_t* red6, const uint8_t* blue6) {
    if (!c || !red6 || !blue6) return fail(TSD_E_INVALID, "NULL argument");
    CU(cudaSetDevice(c->device));
    const int D = c->cfg.window, npx = D * D;
    ScoreTemplates* h = new ScoreTemplates();
    memset(h, 0, sizeof *h);
    for (int k = 0; k < 12; k++) {
        const uint8_t* t = (k < 6 ? red6 : blue6) + (size_t)(k % 6) * npx;
        int T = 0;
        for (int p = 0; p < npx; p++) {
            // matrix2 = template // 255 (DET:552): only the value 255 counts
            if (t[p] == 255) { h->bits[k][p >> 5] |= 1u << (p & 31); T++; }
            else if (t[p] != 0) { delete h; return fail(TSD_E_INVALID, "template %d pixel %d = %d, expected 0 or 255", k, p, t[p]); }
        }
        const double shape = (double)npx;
        const int tn = npx - T;                              // FP == 0 always (mask*template wraps to {0,1}, DET:254)
        const bool degenerate = (shape + shape * 0.01 >= (double)tn) && ((double)tn >= shape - shape * 0.01);   // DET:563-565
        for (int tp = 0; tp <= npx; tp++) {
            int v = 0;
            if (!degenerate && tp <= T && (tp + T) > 0) v = round2_hundredths((2.0 * tp) / (double)((2 * tp) + 0 + (T - tp)));
            h->lut[k][tp] = (uint8_t)v;
        }
    }
    // the batch enqueued last may still be running on an internal stream (overlap mode) and reading d_tmpl: order the upload after it
    if (join_pending(c) != TSD_OK) { delete h; return TSD_E_CUDA; }
    cudaError_t e = cudaMemcpyAsync(c->d_tmpl, h, sizeof *h, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    delete h;
    if (e != cudaSuccess) return fail(TSD_E_CUDA, "template upload: %s", cudaGetErrorString(e));
    c->have_templates = true;
    c->tmpl_D = D;
    return TSD_OK;
}

int tsd_set_similarity_table(tsd_ctx* c, const double* f, int n) {
    if (!c || !f || n < 2 || n > (1 << 30)) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    // the kernel treats d2 >= n as "no action": require f(n-1) small enough that sqrt(f) < tol*merge_factor for both passes
    if (sqrt(f[n - 1]) >= c->cfg.coord_tol * c->cfg.merge_factor) return fail(TSD_E_INVALID, "similarity table too short: f(%d)=%g", n - 1, f[n - 1]);
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_simtab) CU(cudaFree(c->d_simtab));
    c->d_simtab = nullptr;
    CU(cudaMalloc(&c->d_simtab, sizeof(double) * n));
    CU(cudaMemcpy(c->d_simtab, f, sizeof(double) * n, cudaMemcpyHostToDevice));
    c->simtab_n = n;
    c->h_simtab.assign(f, f + n);
    c->gen++;
    return TSD_OK;
}

int tsd_set_lda(tsd_ctx* c, const double* W, const double* b, int nfeat) {
    if (!c || !W || !b || nfeat < 1 || nfeat > 4096) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    // k8_lda_kernel stages W in dynamic shared memory: nfeat * 48 B, 192 KB at 4096 features (above 48 KB it needs the opt-in)
    TRY(allow_dynamic_smem(c, (const void*)k8_lda_kernel, (size_t)nfeat * 6 * sizeof(double), "k8_lda"));
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    if (c->d_ldaW) cudaFree(c->d_ldaW);
    if (c->d_ldab) cudaFree(c->d_ldab);
    CU(cudaMalloc(&c->d_ldaW, sizeof(double) * nfeat * 6));
    CU(cudaMalloc(&c->d_ldab, sizeof(double) * 6));
    CU(cudaMemcpy(c->d_ldaW, W, sizeof(double) * nfeat * 6, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_ldab, b, sizeof(double) * 6, cudaMemcpyHostToDevice));
    c->lda_nfeat = nfeat;
    c->gen++;
    return TSD_OK;
}

int tsd_set_knn(tsd_ctx* c, const double* xbar, const double* scalings, int nfeat, const double* Ztrain, const int32_t* ytrain,
                int ntrain, int k) {
    if (!c || !xbar || !scalings || !Ztrain || !ytrain || nfeat < 1 || ntrain < 1 || k < 1 || k > kKnnMaxK)
        return fail(TSD_E_INVALID, "bad argument (k must be 1..%d)", kKnnMaxK);
    for (int t = 0; t < ntrain; t++)                         // k8_knn_kernel votes into 16 label counters
        if (ytrain[t] < 0 || ytrain[t] >= kKnnMaxLabels)
            return fail(TSD_E_INVALID, "ytrain[%d] = %d, labels must be 0..%d", t, ytrain[t], kKnnMaxLabels - 1);
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    void* old[] = {c->d_xbar, c->d_scal, c->d_Zt, c->d_yt};
    for (void* p : old) if (p) cudaFree(p);
    CU(cudaMalloc(&c->d_xbar, sizeof(double) * nfeat));
    CU(cudaMalloc(&c->d_scal, sizeof(double) * nfeat * 6));
    CU(cudaMalloc(&c->d_Zt, sizeof(double) * (size_t)ntrain * 6));
    CU(cudaMalloc(&c->d_yt, sizeof(int32_t) * ntrain));
    CU(cudaMemcpy(c->d_xbar, xbar, sizeof(double) * nfeat, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_scal, scalings, sizeof(double) * nfeat * 6, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_Zt, Ztrain, sizeof(double) * (size_t)ntrain * 6, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_yt, ytrain, sizeof(int32_t) * ntrain, cudaMemcpyHostToDevice));
    c->knn_nfeat = nfeat; c->knn_ntrain = ntrain; c->knn_k = k;
    c->gen++;
    return TSD_OK;
}

}  // extern "C"

// ---- staging helpers for host-pointer calls ----------------------------------------------------------------------
struct Stage {                                               // stream-ordered temporaries, freed on destruction
    tsd_ctx* c;
    std::vector<void*> ptrs;
    explicit Stage(tsd_ctx* ctx) : c(ctx) { join_pending(ctx); }
    ~Stage() { for (void* p : ptrs) cudaFreeAsync(p, c->stream); }
    int alloc(void** p, size_t bytes) {
        CU(cudaMallocAsync(p, bytes ? bytes : 1, c->stream));
        ptrs.push_back(*p);
        return TSD_OK;
    }
    int in(const void* host, size_t bytes, void** dev) {
        TRY(alloc(dev, bytes));
        if (bytes) CU(cudaMemcpyAsync(*dev, host, bytes, cudaMemcpyHostToDevice, c->stream));
        return TSD_OK;
    }
    int out(void* host, const void* dev, size_t bytes) {
        if (bytes) CU(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, c->stream));
        return TSD_OK;
    }
};

static HsvBounds bounds_of(const tsd_config& cfg) {
    HsvBounds hb;
    memcpy(hb.red_lo, cfg.red_lo, 6); memcpy(hb.red_hi, cfg.red_hi, 6);
    memcpy(hb.blue_lo, cfg.blue_lo, 3); memcpy(hb.blue_hi, cfg.blue_hi, 3);
    return hb;
}

// ---- device-pointer implementations --------------------------------------------------------------------------------
static int dev_expand(tsd_ctx* c, const int32_t* boxes, int n, double enlarge, int32_t* coords, uint8_t* valid) {
    if (n == 0) return TSD_OK;
    k1_expand_kernel<<<cdiv(n, 256), 256, 0, c->cur>>>((const int4*)boxes, n, enlarge - 1.0, c->cfg.aspect_lo, c->cfg.aspect_hi, (int4*)coords, valid);
    return check_launch(c, "k1_expand");
}

// out_stride = bytes between output windows: D*D*ch (public packed layout) or win_stride() (internal, zero padded).
// nframes = frames behind `frames` (the TMA variant's tensor map needs the extent; 0 = unknown: direct gather).
static int dev_crop_resize(tsd_ctx* c, const uint8_t* frames, int H, int W, int64_t rs, int64_t fs, int ch, const int32_t* coords,
                           const int32_t* win_frame, const int32_t* n_ptr, int n_max, int D, uint8_t* windows, int out_stride, int nframes = 0) {
    if (n_max == 0) return TSD_OK;
    if (rs * (int64_t)H >= ((int64_t)1 << 31)) return fail(TSD_E_INVALID, "a frame must span less than 2 GiB (row offsets are 32-bit)");
    const int g4_all = cdiv(n_max, 4);                       // one window per warp (the generic kernel does not loop)
    int g4 = g4_all;
    if (c->k2_grid > 0 && g4 > c->k2_grid * c->sm_count) g4 = c->k2_grid * c->sm_count;     // persistent warps (the v2 / TMA kernels stride over the windows)
    int skip_tma = 0;
#define K2_ARGS frames, H, W, rs, fs, (const int4*)coords, win_frame, n_ptr, n_max
    // TSD_K2=tma: ROI staged by the Tensor Memory Accelerator (internal 16-byte window layout, BGR, D = 25 / 32, TMA-legal frame layout)
    if (c->k2_tma && ch == 3 && (D == 25 || D == 32) && nframes > 0 && out_stride % 16 == 0 && ((uintptr_t)windows % 16) == 0) {
        K2TensorMaps maps;
        if (k2_build_tensor_maps(&maps, frames, nframes, H, W, rs, fs)) {
            const size_t smem = (size_t)kTmaWarps * tma_warp_bytes(D) + 128;
            if (!c->attr_k2tma) {
                CU(cudaFuncSetAttribute(k2_crop_resize_tma_kernel<25>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kTmaWarps * tma_warp_bytes(25) + 128)));
                CU(cudaFuncSetAttribute(k2_crop_resize_tma_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kTmaWarps * tma_warp_bytes(32) + 128)));
                CU(cudaFuncSetAttribute(k2_crop_resize_tma_kernel<25>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                CU(cudaFuncSetAttribute(k2_crop_resize_tma_kernel<32>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                c->attr_k2tma = true;
            }
            // one window per warp; the crops that do not fit the staging buffer are left to the gather kernel launched right after
            if (D == 25) k2_crop_resize_tma_kernel<25><<<g4, kTmaWarps * 32, smem, c->cur>>>(maps, K2_ARGS, windows, out_stride);
            else k2_crop_resize_tma_kernel<32><<<g4, kTmaWarps * 32, smem, c->cur>>>(maps, K2_ARGS, windows, out_stride);
            TRY(check_launch(c, "k2_crop_resize_tma"));
            skip_tma = 1;
        }
    }
    // aligned 32-bit tap loads need 4-byte aligned frames and strides and the number of frames (the last row of the last frame keeps byte loads)
    const int wide_last = (nframes > 0 && ((uintptr_t)frames % 4) == 0 && rs % 4 == 0 && fs % 4 == 0) ? nframes - 1 : -2;
    if (ch == 3 && D == 25) k2_crop_resize_v2_kernel<3, 25><<<g4, 128, 0, c->cur>>>(K2_ARGS, windows, out_stride, skip_tma, wide_last);
    else if (ch == 3 && D == 32) k2_crop_resize_v2_kernel<3, 32><<<g4, 128, 0, c->cur>>>(K2_ARGS, windows, out_stride, skip_tma, wide_last);
    else if (ch == 1 && D == 25) k2_crop_resize_v2_kernel<1, 25><<<g4, 128, 0, c->cur>>>(K2_ARGS, windows, out_stride, 0, -2);
    else if (ch == 1 && D == 32) k2_crop_resize_v2_kernel<1, 32><<<g4, 128, 0, c->cur>>>(K2_ARGS, windows, out_stride, 0, -2);
    else if (ch == 3) k2_crop_resize_kernel<3><<<g4_all, 128, 0, c->cur>>>(K2_ARGS, D, windows, out_stride);      // other window sizes: generic kernel
    else k2_crop_resize_kernel<1><<<g4_all, 128, 0, c->cur>>>(K2_ARGS, D, windows, out_stride);
#undef K2_ARGS
    return check_launch(c, "k2_crop_resize");
}

// words per bit row of the pair-class matrix for frames of up to max_n windows (the warp fold handles at most 1024)
static inline int pair_row_words(int max_n) {
    if (max_n > 1024) max_n = 1024;
    return ((max_n > 1 ? max_n : 1) + 31) / 32;
}

// K1 count (+ scan by its last CTA) + compact -> coords/win_frame/win_offsets in context scratch or caller buffers
static int dev_windows_index(tsd_ctx* c, const int32_t* boxes, const int32_t* box_offsets, int nframes, int H, int W, double enlarge,
                             int32_t* counts, int32_t* win_offsets, int32_t* coords, int32_t* win_frame) {
    const double pm1 = enlarge - 1.0;
    k1_count_kernel<<<cdiv((int64_t)nframes * 32, 128), 128, 0, c->cur>>>((const int4*)boxes, box_offsets, nframes, H, W, pm1, c->cfg.aspect_lo, c->cfg.aspect_hi, counts,
                                                                           win_offsets, c->d_tickets + c->ticket_base);
    TRY(check_launch(c, "k1_count"));
    k1_compact_kernel<<<cdiv((int64_t)nframes * 32, 128), 128, 0, c->cur>>>((const int4*)boxes, box_offsets, nframes, H, W, pm1, c->cfg.aspect_lo, c->cfg.aspect_hi, win_offsets, (int4*)coords, win_frame);
    return check_launch(c, "k1_compact");
}

// ws = bytes between windows (packed or padded); entries are written with stride ent_stride(npx) words
static int dev_hist(tsd_ctx* c, const uint8_t* windows, const int32_t* n_ptr, int n_max, int npx, int ws, uint32_t* entries, WinMeta* meta,
                    float* E_T, int64_t e_stride) {
    if (n_max == 0) return TSD_OK;
#define HIST_ARGS windows, n_ptr, n_max, npx, ws, ent_stride(npx), c->d_tab, entries, meta, E_T, e_stride
    if (npx <= 640) {
        int grid = cdiv(n_max, 4);
        if (grid > c->sm_count * TSD_HIST_GRID) grid = c->sm_count * TSD_HIST_GRID;
        k5_hist_kernel<640, 4, TSD_HIST_MINB, HsvLut><<<grid, 128, sizeof(HistKSmem<640, 4, HsvLut>), c->cur>>>(HIST_ARGS);
    } else {
        int grid = cdiv(n_max, 3);
        if (grid > c->sm_count * TSD_HIST_GRID) grid = c->sm_count * TSD_HIST_GRID;
        k5_hist_kernel<1024, 3, 1, HsvLut><<<grid, 96, sizeof(HistKSmem<1024, 3, HsvLut>), c->cur>>>(HIST_ARGS);
    }
#undef HIST_ARGS
    return check_launch(c, "k5_hist");
}

// K5: both (or one) passes of cleanDuplicatedDetections.  max_n = upper bound of windows per frame (host-known), ncap = total
// windows (rows of the pair-class bit matrix).  max_n <= 1024: all-pairs classification (k5_gram / k5_pairs) + one warp per frame
// (k5_fold_warp); larger frames: the general block-synchronous fold (k5_fold_kernel).
// The fold of one batch: frames of up to kFoldCtaMin windows by one warp each (k5_fold_warp), larger ones (<= 1024) by one CTA each
// (k5_fold_cta); both walk the same longest-first order list with their own work counter.
template <int CAP>
static int launch_folds(tsd_ctx* c, int variant, const FoldParams& P, int nframes, uint32_t* M, int RW, int cut, const int32_t* cost, int max_n) {
    const int warps = kFoldWarps;
    const size_t smem = ((sizeof(HsvLut) + 15) & ~(size_t)15) + (size_t)warps * sizeof(FoldWarpSmem<256, CAP>);
    const size_t smem_cta = sizeof(FoldCtaSmem<CAP>);
    int& per_sm = c->fold_per_sm[variant];
    int& per_sm_cta = c->fold_per_sm[2 + variant];
    if (!per_sm) {
        CU(cudaFuncSetAttribute(k5_fold_warp_kernel<256, CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CU(cudaFuncSetAttribute(k5_fold_warp_kernel<256, CAP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k5_fold_warp_kernel<256, CAP>, warps * 32, smem));
        if (per_sm < 1) per_sm = 1;
        CU(cudaFuncSetAttribute(k5_fold_cta_kernel<CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cta));
        CU(cudaFuncSetAttribute(k5_fold_cta_kernel<CAP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_cta, k5_fold_cta_kernel<CAP>, kFoldCtaWarps * 32, smem_cta));
        if (per_sm_cta < 1) per_sm_cta = 1;
        if (getenv("TSD_DEBUG")) fprintf(stderr, "[tsd] k5_fold_warp<256,%d>: %zu B shared memory per CTA, %d CTAs per SM; k5_fold_cta: %zu B, %d per SM\n", CAP, smem, per_sm, smem_cta, per_sm_cta);
    }
    // longest-first frame order + the two work counters + the costs in that order (context scratch: [nframes] order, [2] counters,
    // [nframes] costs)
    int32_t* order = (int32_t*)c->b_order.p + 2 * c->order_off;
    int32_t* counter = order + nframes;
    int32_t* cost_sorted = counter + 2;
    k5_order_kernel<<<1, 1024, 0, c->cur>>>(cost, P.offsets, nframes, order, counter, cost_sorted);
    TRY(check_launch(c, "k5_order"));
    // frames predicted to merge often go to the CTA fold too (batches large enough for a straggler to matter)
    const int cost_min = (cost && nframes >= 256) ? c->fold_cta_cost : 0;
    int grid = cdiv(nframes, warps);
    // Resident fold CTAs per SM: each holds 16 K registers and ~56 KB of shared memory, so the four that fit take the WHOLE SM and the
    // kernels of the other batch (two-slot overlap) cannot run beside them; a cap leaves room (the fold is bound by latency, not by
    // the number of its warps: one batch needs ~1100 warp-milliseconds spread over the ~2.6 ms the other batch's kernels take).
    const int cap_sm = (c->fold_per_sm_cap > 0 && c->fold_per_sm_cap < per_sm) ? c->fold_per_sm_cap : per_sm;
    if (grid > cap_sm * c->sm_count) grid = cap_sm * c->sm_count;
    k5_fold_warp_kernel<256, CAP><<<grid, warps * 32, smem, c->cur>>>(P, nframes, M, RW, cut, order, counter, kFoldCtaMin, cost_sorted, cost_min);
    TRY(check_launch(c, "k5_fold_warp"));
    if (max_n > kFoldCtaMin || cost_min > 0) {
        grid = nframes < per_sm_cta * c->sm_count ? nframes : per_sm_cta * c->sm_count;
        k5_fold_cta_kernel<CAP><<<grid, kFoldCtaWarps * 32, smem_cta, c->cur>>>(P, nframes, M, RW, cut, order, counter + 1, kFoldCtaMin, cost_sorted, cost_min);
        TRY(check_launch(c, "k5_fold_cta"));
    }
    return TSD_OK;
}

// M = the batch's rows of the pair-class bit matrix (2 * RW words per window, RW = words per bit row for max_n windows per frame);
// todo = the batch's work list for k5_pairs ([count, items ...], todo_capacity(nframes, max_n) ints).
static inline size_t todo_capacity(int nframes, int max_n) {
    const int nbk = (std::min(max_n, 1024) + kGramBM - 1) / kGramBM;
    return (size_t)nframes * std::max(1, nbk * (nbk + 1) / 2) + 2;
}

static int dev_fold(tsd_ctx* c, uint8_t* windows, int ws, int32_t* coords, uint32_t* entries, WinMeta* meta, const int32_t* offsets, int nframes,
                    int npx, int do_hist, int do_coords, double hist_tol, double coord_tol, int32_t* list, uint8_t* flags, int32_t* out_count,
                    int max_n, uint32_t* M, int32_t* todo, float* E_T, int64_t e_stride, int32_t* surv_offsets, cudaEvent_t front_done = nullptr) {
    FoldParams P;
    P.windows = windows; P.coords = (int4*)coords; P.entries = entries; P.meta = meta; P.offsets = offsets;
    P.list = list; P.flags = flags; P.out_count = out_count; P.simtab = c->d_simtab; P.simtab_n = c->simtab_n; P.tab = c->d_tab;
    P.npx = npx; P.ws = ws; P.es = ent_stride(npx); P.do_hist = do_hist; P.do_coords = do_coords;
    P.E_T = E_T; P.e_stride = e_stride;
    P.hist_tol = hist_tol; P.hist_lo = hist_tol * c->cfg.merge_factor;      // tolerance * 0.8823 in f64 (DET:217)
    P.coord_tol = coord_tol; P.coord_lo = coord_tol * c->cfg.merge_factor;
    if (do_coords) TRY(check_simtab(c, P.coord_lo, "tol * merge_factor ="));
    if (nframes == 0) { if (surv_offsets) CU(cudaMemsetAsync(surv_offsets, 0, 4, c->cur)); return TSD_OK; }
    // max_n is only an upper bound (raw boxes per frame); frames with more than 1024 aspect-passing windows are flagged by
    // the warp-per-frame fold (out_count = -1) and redone by the general block-synchronous fold below
    const int RW = pair_row_words(max_n);
    if (max_n > 1024) max_n = 1024;
    // Corner similarity can only act when sqrt(f1 f2) >= coord_lo, i.e. both f >= coord_lo^2: squared distances at or
    // beyond `cut` are class 0 without a table lookup (f is non-increasing in d2).
    int cut = c->simtab_n;
    {
        const double thr = P.coord_lo * P.coord_lo * (1.0 - 1e-9);
        int lo_i = 0, hi_i = c->simtab_n;                    // first index with f < thr
        while (lo_i < hi_i) { int mid = (lo_i + hi_i) / 2; if (c->h_simtab[mid] < thr) hi_i = mid; else lo_i = mid + 1; }
        cut = lo_i > 0 ? lo_i : 1;
    }
    int32_t* cost = nullptr;
    if (do_hist) {
        cost = out_count;                                    // [nframes] scratch until the fold writes the survivor counts (order is built first)
        CU(cudaMemsetAsync(cost, 0, (size_t)nframes * 4, c->cur));
        // frames of up to kGramBM windows: Gram matrix on the tensor cores, one CTA per frame (k5_gram); larger frames (<= 1024): one
        // CTA per pair of 128-row blocks (k5_gram_big); what they leave over (flat frames), and everything with TSD_GRAM=0: k5_pairs
        int32_t* gram_done = nullptr;
        if (c->use_gram) {
            if (!c->attr_gram) {
                CU(cudaFuncSetAttribute(k5_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(GramSmem)));
                CU(cudaFuncSetAttribute(k5_gram_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                CU(cudaFuncSetAttribute(k5_gram_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(GramBigSmem)));
                CU(cudaFuncSetAttribute(k5_gram_big_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
                c->attr_gram = true;
            }
            gram_done = todo;                                // [count, items ...] for k5_pairs; behind it the same for k5_gram_big
            int32_t* big = todo + todo_capacity(nframes, max_n);
            CU(cudaMemsetAsync(gram_done, 0, 4, c->cur));
            CU(cudaMemsetAsync(big, 0, 4, c->cur));
            k5_gram_kernel<<<nframes, kGramWarps * 32, sizeof(GramSmem), c->cur>>>(entries, meta, E_T, e_stride, offsets, nframes, P.es, RW, P.hist_tol,
                                                                                   P.hist_lo, M, cost, gram_done, big, 2 * c->sm_count);
            TRY(check_launch(c, "k5_gram"));
            if (max_n > kGramBM) {                           // persistent CTAs (one per SM: 148 KB of shared memory) walk the list k5_gram wrote
                k5_gram_big_kernel<<<c->sm_count, kBigWarps * 32, sizeof(GramBigSmem), c->cur>>>(entries, meta, E_T, e_stride, offsets, nframes, P.es, RW,
                                                                                                 P.hist_tol, P.hist_lo, M, cost, gram_done, big);
                TRY(check_launch(c, "k5_gram_big"));
            }
        }
        {
            const int tiles = (max_n + kPairWarps - 1) / kPairWarps;
            const size_t psm = kPairWarps * kDenseLen * 2;
            // with a todo list (what the Gram kernels left over) a grid of resident CTAs walks it; else one CTA per (frame, tile)
            const int pgrid = gram_done ? (int)std::min<int64_t>((int64_t)nframes * tiles, (int64_t)c->sm_count * 16) : nframes * tiles;
            if (!c->attr_pairs) {
                CU(cudaFuncSetAttribute(k5_pairs_kernel<1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
                c->attr_pairs = true;
            }
            k5_pairs_kernel<1, 8><<<pgrid, kPairWarps * 32, psm, c->cur>>>(entries, meta, E_T, e_stride, offsets, nframes, P.es, RW, tiles,
                                                                             P.hist_tol, P.hist_lo, M, cost, gram_done);
            TRY(check_launch(c, "k5_pairs"));
        }
        mark(c, "k5_pairs");
    }
    if (front_done) TRY(ev_record(c, front_done));           // the next batch's front half may start (enqueue_chain)
    TRY(npx <= 640 ? launch_folds<640>(c, 0, P, nframes, M, RW, cut, cost, max_n) : launch_folds<1024>(c, 1, P, nframes, M, RW, cut, cost, max_n));
    // Frames the warp fold flagged (more windows than its variant or the caller's max_boxes_per_frame bound allows) are redone by the
    // general fold.  Always launched: it costs ~10 us when nothing is flagged and makes a too-small caller bound harmless.
    // (its CTAs stride over the frames: a few per SM check the flags of a large batch in ~5 us instead of one CTA per frame in ~20)
    k5_fold_kernel<<<std::min(nframes, 4 * c->sm_count), kFoldThreads, 0, c->cur>>>(P, nframes, 1, surv_offsets, c->d_tickets + c->ticket_base + 1);
    return check_launch(c, "k5_fold");
}

// ---------------------------------------------------------------------------------------------------------------
extern "C" {

int tsd_expand_boxes(tsd_ctx* c, const int32_t* boxes, int nboxes, double enlarge, int32_t* coords, uint8_t* valid, int mem) {
    if (!c || nboxes < 0 || (nboxes && (!boxes || !coords || !valid))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (mem == TSD_MEM_DEVICE) return dev_expand(c, boxes, nboxes, enlarge, coords, valid);
    Stage s(c);
    void *db, *dc, *dv;
    TRY(s.in(boxes, (size_t)nboxes * 16, &db));
    TRY(s.alloc(&dc, (size_t)nboxes * 16));
    TRY(s.alloc(&dv, (size_t)nboxes));
    TRY(dev_expand(c, (int32_t*)db, nboxes, enlarge, (int32_t*)dc, (uint8_t*)dv));
    TRY(s.out(coords, dc, (size_t)nboxes * 16));
    TRY(s.out(valid, dv, (size_t)nboxes));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_crop_resize(tsd_ctx* c, const uint8_t* frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride, int channels,
                    const int32_t* coords, const int32_t* win_frame, int n, int D, uint8_t* windows, int mem) {
    if (!c || !frames || nframes < 1 || H < 1 || W < 1 || n < 0 || (channels != 1 && channels != 3) || D < 2 || D > kMaxD)
        return fail(TSD_E_INVALID, "bad argument");
    if (row_stride < (int64_t)W * channels || frame_stride < row_stride * (H - 1) + (int64_t)W * channels) return fail(TSD_E_INVALID, "bad strides");
    if (n && (!coords || !win_frame || !windows)) return fail(TSD_E_INVALID, "NULL argument");
    CU(cudaSetDevice(c->device));
    // Device pointers: the kernel zero-fills a window whose clipped crop is empty (cv2.resize would raise; the chain never asks for
    // one: K1 drops such boxes).  Host pointers are checked here, like the reference's own exceptions.
    if (mem == TSD_MEM_DEVICE) return dev_crop_resize(c, frames, H, W, row_stride, frame_stride, channels, coords, win_frame, nullptr, n, D, windows, D * D * channels, nframes);
    for (int i = 0; i < n; i++) {
        const int32_t* q = coords + 4 * (size_t)i;
        if (win_frame[i] < 0 || win_frame[i] >= nframes) return fail(TSD_E_INVALID, "window %d: frame %d not in [0,%d)", i, win_frame[i], nframes);
        if (q[0] < 0 || q[1] < 0 || q[2] < 0 || q[3] < 0) return fail(TSD_E_INVALID, "window %d: negative coordinate (numpy slicing would wrap around)", i);
        if (std::min(q[2], W) <= std::min(q[0], W) || std::min(q[3], H) <= std::min(q[1], H))
            return fail(TSD_E_INVALID, "window %d: empty crop after clipping to the frame (cv2.resize would raise)", i);
    }
    Stage s(c);
    void *df, *dc, *dwf, *dw;
    TRY(s.in(frames, (size_t)frame_stride * (nframes - 1) + (size_t)row_stride * (H - 1) + (size_t)W * channels, &df));
    TRY(s.in(coords, (size_t)n * 16, &dc));
    TRY(s.in(win_frame, (size_t)n * 4, &dwf));
    TRY(s.alloc(&dw, (size_t)n * D * D * channels));
    TRY(dev_crop_resize(c, (uint8_t*)df, H, W, row_stride, frame_stride, channels, (int32_t*)dc, (int32_t*)dwf, nullptr, n, D, (uint8_t*)dw, D * D * channels, nframes));
    TRY(s.out(windows, dw, (size_t)n * D * D * channels));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_windows(tsd_ctx* c, const uint8_t* frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride,
                const int32_t* boxes, const int32_t* box_offsets, double enlarge, int D, uint8_t* windows, int32_t* coords,
                int32_t* win_offsets, int32_t* total, int mem) {
    if (!c || !frames || !box_offsets || !win_offsets || nframes < 1 || H < 1 || W < 1 || D < 2 || D > kMaxD) return fail(TSD_E_INVALID, "bad argument");
    if (row_stride < (int64_t)W * 3 || frame_stride < row_stride * (H - 1) + (int64_t)W * 3) return fail(TSD_E_INVALID, "bad strides");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "tsd_windows takes host pointers; use tsd_enqueue_frames for device-resident batches");
    CU(cudaSetDevice(c->device));
    const int nb = box_offsets[nframes];
    if (nb < 0 || (nb && !boxes)) return fail(TSD_E_INVALID, "bad boxes");
    for (int f = 0; f < nframes; f++) if (box_offsets[f + 1] < box_offsets[f]) return fail(TSD_E_INVALID, "box_offsets must not decrease (frame %d)", f);
    Stage s(c);
    void *df, *db, *dbo, *dcnt, *dwo, *dc, *dwf, *dw;
    TRY(s.in(frames, (size_t)frame_stride * (nframes - 1) + (size_t)row_stride * (H - 1) + (size_t)W * 3, &df));
    TRY(s.in(boxes, (size_t)nb * 16, &db));
    TRY(s.in(box_offsets, (size_t)(nframes + 1) * 4, &dbo));
    TRY(s.alloc(&dcnt, (size_t)nframes * 4));
    TRY(s.alloc(&dwo, (size_t)(nframes + 1) * 4));
    TRY(s.alloc(&dc, (size_t)nb * 16));
    TRY(s.alloc(&dwf, (size_t)nb * 4));
    TRY(s.alloc(&dw, (size_t)nb * D * D * 3));
    TRY(dev_windows_index(c, (int32_t*)db, (int32_t*)dbo, nframes, H, W, enlarge, (int32_t*)dcnt, (int32_t*)dwo, (int32_t*)dc, (int32_t*)dwf));
    TRY(dev_crop_resize(c, (uint8_t*)df, H, W, row_stride, frame_stride, 3, (int32_t*)dc, (int32_t*)dwf, (int32_t*)dwo + nframes, nb, D, (uint8_t*)dw, D * D * 3, nframes));
    TRY(s.out(win_offsets, dwo, (size_t)(nframes + 1) * 4));
    CU(cudaStreamSynchronize(c->stream));
    const int tot = win_offsets[nframes];
    if (total) *total = tot;
    if (tot) {
        if (!windows || !coords) return fail(TSD_E_INVALID, "NULL output");
        TRY(s.out(windows, dw, (size_t)tot * D * D * 3));
        TRY(s.out(coords, dc, (size_t)tot * 16));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

int tsd_dedup(tsd_ctx* c, const uint8_t* windows, const int32_t* coords, const int32_t* offsets, int nframes, int D, int by_coords,
              double tol, uint8_t* out_windows, int32_t* out_coords, int32_t* out_offsets, int32_t* total_out, int mem) {
    if (!c || !offsets || !out_offsets || nframes < 0 || D < 2 || D > kMaxD) return fail(TSD_E_INVALID, "bad argument");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "tsd_dedup takes host pointers; use tsd_enqueue_frames for device-resident batches");
    CU(cudaSetDevice(c->device));
    const int n = offsets[nframes], npx = D * D, nbytes = npx * 3, ws = win_stride(npx, 3), es = ent_stride(npx);
    if (n && (!windows || !coords)) return fail(TSD_E_INVALID, "NULL argument");
    for (int64_t i = 0; i < (int64_t)n * 4; i++)             // (the corner distances are evaluated in 32-bit arithmetic)
        if (coords[i] < 0 || coords[i] >= (1 << 30)) return fail(TSD_E_INVALID, "coordinate %d of window %d out of range [0, 2^30)", coords[i], (int)(i / 4));
    Stage s(c);
    void *dw, *dc, *doff, *dent, *dmeta, *dlist, *dflags, *dcnt, *dooff, *dow, *doc, *den;
    TRY(s.alloc(&dw, (size_t)n * ws));                       // internal layout: 16-byte aligned windows, zero pad
    if (n) {
        CU(cudaMemsetAsync(dw, 0, (size_t)n * ws, c->stream));
        CU(cudaMemcpy2DAsync(dw, ws, windows, nbytes, nbytes, n, cudaMemcpyHostToDevice, c->stream));
    }
    TRY(s.in(coords, (size_t)n * 16, &dc));
    TRY(s.in(offsets, (size_t)(nframes + 1) * 4, &doff));
    TRY(s.alloc(&dent, (size_t)n * es * 4));
    TRY(s.alloc(&dmeta, (size_t)n * sizeof(WinMeta)));
    TRY(s.alloc(&dlist, (size_t)n * 4));
    TRY(s.alloc(&dflags, (size_t)n));
    TRY(s.alloc(&den, (size_t)(n > 0 ? n : 1) * kEnergyRows * 4));
    TRY(s.alloc(&dcnt, (size_t)(nframes + 1) * 4));
    TRY(s.alloc(&dooff, (size_t)(nframes + 1) * 4));
    TRY(s.alloc(&dow, (size_t)n * nbytes));
    TRY(s.alloc(&doc, (size_t)n * 16));
    if (n) {
        if (by_coords) {
            k5_hash_kernel<<<cdiv((int64_t)n * 32, 128), 128, 0, c->cur>>>((uint8_t*)dw, n, npx, ws, (WinMeta*)dmeta);
            TRY(check_launch(c, "k5_hash"));
        } else {
            TRY(dev_hist(c, (uint8_t*)dw, nullptr, n, npx, ws, (uint32_t*)dent, (WinMeta*)dmeta, (float*)den, n));
        }
    }
    int max_n = 0;
    for (int f = 0; f < nframes; f++) max_n = offsets[f + 1] - offsets[f] > max_n ? offsets[f + 1] - offsets[f] : max_n;
    c->order_off = 0;
    TRY(ensure(c, c->b_pairs, (size_t)(n > 0 ? n : 1) * 2 * pair_row_words(max_n) * sizeof(uint32_t)));
    TRY(ensure(c, c->b_gramdone, 2 * todo_capacity(nframes, max_n) * 4));
    TRY(ensure(c, c->b_order, (size_t)(2 * nframes + 4) * 4));
    TRY(dev_fold(c, (uint8_t*)dw, ws, (int32_t*)dc, (uint32_t*)dent, (WinMeta*)dmeta, (int32_t*)doff, nframes, npx, !by_coords, by_coords,
                 tol, tol, (int32_t*)dlist, (uint8_t*)dflags, (int32_t*)dcnt, max_n, (uint32_t*)c->b_pairs.p, (int32_t*)c->b_gramdone.p, (float*)den, n, (int32_t*)dooff));
    if (nframes) {
        k5_gather_kernel<<<nframes, 128, 0, c->cur>>>((uint8_t*)dw, (int4*)dc, (int32_t*)doff, (int32_t*)dlist, (int32_t*)dooff, nframes, nbytes, ws,
                                                         (uint8_t*)dow, (int4*)doc, nullptr);
        TRY(check_launch(c, "k5_gather"));
    }
    TRY(s.out(out_offsets, dooff, (size_t)(nframes + 1) * 4));
    CU(cudaStreamSynchronize(c->stream));
    const int tot = out_offsets[nframes];
    if (total_out) *total_out = tot;
    if (tot) {
        if (!out_windows || !out_coords) return fail(TSD_E_INVALID, "NULL output");
        TRY(s.out(out_windows, dow, (size_t)tot * nbytes));
        TRY(s.out(out_coords, doc, (size_t)tot * 16));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

int tsd_hist(tsd_ctx* c, const uint8_t* windows, int n, int D, float* hist, int mem) {
    if (!c || n < 0 || D < 2 || D > kMaxD || (n && (!windows || !hist))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    const int npx = D * D;
    Stage s(c);
    void *dw = (void*)windows, *dh = (void*)hist, *dent, *dmeta;
    if (mem == TSD_MEM_HOST) { TRY(s.in(windows, (size_t)n * npx * 3, &dw)); TRY(s.alloc(&dh, (size_t)n * kHistBins * 4)); }
    TRY(s.alloc(&dent, (size_t)n * ent_stride(npx) * 4));
    TRY(s.alloc(&dmeta, (size_t)n * sizeof(WinMeta)));
    TRY(dev_hist(c, (uint8_t*)dw, nullptr, n, npx, npx * 3, (uint32_t*)dent, (WinMeta*)dmeta, nullptr, 0));      // public layout: packed windows
    hist_dense_kernel<<<n, 256, 0, c->cur>>>((uint32_t*)dent, (WinMeta*)dmeta, n, ent_stride(npx), (float*)dh);
    TRY(check_launch(c, "hist_dense"));
    if (mem == TSD_MEM_HOST) { TRY(s.out(hist, dh, (size_t)n * kHistBins * 4)); CU(cudaStreamSynchronize(c->stream)); }
    return TSD_OK;
}

int tsd_color_masks(tsd_ctx* c, const uint8_t* windows, int n, int D, uint8_t* red, uint8_t* blue, int mem) {
    if (!c || n < 0 || D < 1 || (n && (!windows || !red || !blue))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    const int npx = D * D;
    Stage s(c);
    void *dw = (void*)windows, *dr = red, *db = blue;
    if (mem == TSD_MEM_HOST) { TRY(s.in(windows, (size_t)n * npx * 3, &dw)); TRY(s.alloc(&dr, (size_t)n * npx)); TRY(s.alloc(&db, (size_t)n * npx)); }
    int grid = cdiv((int64_t)n * 32, 256);
    if (grid > c->sm_count * 8) grid = c->sm_count * 8;
    k3_masks_generic_kernel<<<grid, 256, 0, c->cur>>>((uint8_t*)dw, nullptr, nullptr, n, npx, npx * 3, c->d_tab, bounds_of(c->cfg), (uint8_t*)dr, (uint8_t*)db,
                                                    npx, nullptr);       // public layout: packed windows and masks
    TRY(check_launch(c, "k3_masks"));
    if (mem == TSD_MEM_HOST) { TRY(s.out(red, dr, (size_t)n * npx)); TRY(s.out(blue, db, (size_t)n * npx)); CU(cudaStreamSynchronize(c->stream)); }
    return TSD_OK;
}

int tsd_set_gamma_table(tsd_ctx* c, const uint8_t* table256) {
    if (!c || !table256) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    CU(cudaMemcpyAsync(c->d_gamma, table256, 256, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_preprocess(tsd_ctx* c, const uint8_t* frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride, double clip_limit,
                   int tiles_x, int tiles_y, uint8_t* out, int mem) {
    if (!c || !frames || !out || nframes < 1 || H < 1 || W < 1 || tiles_x < 1 || tiles_y < 1 || tiles_x * tiles_y > 65535)
        return fail(TSD_E_INVALID, "bad argument");
    if (row_stride < (int64_t)W * 3 || frame_stride < row_stride * (H - 1) + (int64_t)W * 3) return fail(TSD_E_INVALID, "bad strides");
    CU(cudaSetDevice(c->device));
    // OpenCV clahe.cpp: if EITHER size is not a multiple of the grid both are extended (BORDER_REFLECT_101) by tiles - size % tiles
    const bool divisible = H % tiles_y == 0 && W % tiles_x == 0;
    const int He = divisible ? H : H + tiles_y - H % tiles_y, We = divisible ? W : W + tiles_x - W % tiles_x;
    const int tw = We / tiles_x, th = He / tiles_y, total = tw * th;
    const float lut_scale = 255.0f / (float)total;
    int clip = 0;
    if (clip_limit > 0.0) { clip = (int)(clip_limit * total / 256); if (clip < 1) clip = 1; }
    const size_t npix = (size_t)nframes * H * W;
    TRY(ensure(c, c->b_pgray, npix));
    TRY(ensure(c, c->b_pluts, (size_t)nframes * tiles_x * tiles_y * 256));
    const uint8_t* d_in = frames;
    uint8_t* d_out = out;
    if (mem == TSD_MEM_HOST) {
        const size_t in_bytes = (size_t)frame_stride * (nframes - 1) + (size_t)row_stride * (H - 1) + (size_t)W * 3;
        TRY(ensure(c, c->b_pin, in_bytes));
        TRY(ensure(c, c->b_pout, npix));
        CU(cudaMemcpyAsync(c->b_pin.p, frames, in_bytes, cudaMemcpyHostToDevice, c->stream));
        d_in = (const uint8_t*)c->b_pin.p; d_out = (uint8_t*)c->b_pout.p;
    }
    // both kernels take the frame from gridDim.y / gridDim.z (at most 65 535): larger batches are launched in frame ranges
    for (int f0 = 0; f0 < nframes; f0 += 65535) {
        const int nf = nframes - f0 < 65535 ? nframes - f0 : 65535;
        uint8_t* gray = (uint8_t*)c->b_pgray.p + (size_t)f0 * H * W;
        uint8_t* luts = (uint8_t*)c->b_pluts.p + (size_t)f0 * tiles_x * tiles_y * 256;
        pre_gray_lut_kernel<<<dim3(tiles_x * tiles_y, nf), 256, 0, c->cur>>>(d_in + (size_t)f0 * frame_stride, H, W, row_stride, frame_stride, tiles_x, tiles_y,
                                                                         tw, th, clip, lut_scale, gray, luts);
        TRY(check_launch(c, "pre_gray_lut"));
        pre_clahe_blur_kernel<<<dim3(cdiv(W, kPreTW), cdiv(H, kPreTH), nf), 256, 0, c->cur>>>(gray, luts, H, W, tiles_x, tiles_y, 1.0f / (float)tw,
                                                                                             1.0f / (float)th, c->d_gamma, d_out + (size_t)f0 * H * W);
        TRY(check_launch(c, "pre_clahe_blur"));
    }
    if (mem == TSD_MEM_HOST) {
        CU(cudaMemcpyAsync(out, d_out, npix, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

int tsd_mean_windows(tsd_ctx* c, const uint8_t* windows, const int32_t* group_offsets, int ngroups, int D, uint8_t* mean_out, int mem) {
    if (!c || !group_offsets || ngroups < 0 || D < 1 || (ngroups && !mean_out)) return fail(TSD_E_INVALID, "bad argument");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "tsd_mean_windows takes host pointers (one-off template building)");
    CU(cudaSetDevice(c->device));
    if (ngroups == 0) return TSD_OK;
    const int n = group_offsets[ngroups], nbytes = D * D * 3;
    if (n && !windows) return fail(TSD_E_INVALID, "NULL argument");
    for (int g = 0; g < ngroups; g++)
        if (group_offsets[g + 1] <= group_offsets[g]) return fail(TSD_E_INVALID, "group %d is empty (the reference would return an all-zero mask; pass at least one window)", g);
    Stage s(c);
    void *dw, *dg, *dm;
    TRY(s.in(windows, (size_t)n * nbytes, &dw));
    TRY(s.in(group_offsets, (size_t)(ngroups + 1) * 4, &dg));
    TRY(s.alloc(&dm, (size_t)ngroups * nbytes));
    mean_windows_kernel<<<ngroups, 32, 0, c->cur>>>((uint8_t*)dw, (int32_t*)dg, ngroups, nbytes, (uint8_t*)dm);
    TRY(check_launch(c, "mean_windows"));
    TRY(s.out(mean_out, dm, (size_t)ngroups * nbytes));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_match_detections(tsd_ctx* c, const int32_t* det, int ndet, const int32_t* gt, const int32_t* gt_offsets, int nframes, double tol,
                         int32_t* status, int32_t* match, int32_t* tally) {
    if (!c || ndet < 0 || nframes < 0 || !gt_offsets || (ndet && (!det || !status || !match)) || (nframes && !tally)) return fail(TSD_E_INVALID, "bad argument");
    if (!c->d_simtab) return fail(TSD_E_STATE, "similarity table not set (tsd_set_similarity_table)");
    TRY(check_simtab(c, tol, "tol ="));                      // eval_match skips ground truths beyond the table
    const int ngt = gt_offsets[nframes];
    if (ngt < 0 || (ngt && !gt)) return fail(TSD_E_INVALID, "bad ground truth");
    for (int i = 0; i < ndet; i++) if (det[6 * i + 5] < 0 || det[6 * i + 5] > 5) return fail(TSD_E_INVALID, "detection %d: type bucket %d not in 0..5", i, det[6 * i + 5]);
    for (int g = 0; g < ngt; g++) if (gt[6 * g + 5] < 0 || gt[6 * g + 5] > 5 || gt[6 * g] < 0 || gt[6 * g] >= nframes) return fail(TSD_E_INVALID, "ground truth %d: bad frame / type bucket", g);
    CU(cudaSetDevice(c->device));
    Stage s(c);
    void *dd = nullptr, *dg = nullptr, *dof, *dst, *dm, *dh, *dt;
    TRY(s.in(det, (size_t)ndet * 24, &dd));
    TRY(s.in(gt, (size_t)ngt * 24, &dg));
    TRY(s.in(gt_offsets, (size_t)(nframes + 1) * 4, &dof));
    TRY(s.alloc(&dst, (size_t)ndet * 4));
    TRY(s.alloc(&dm, (size_t)ndet * 4));
    TRY(s.alloc(&dh, (size_t)ngt));
    TRY(s.alloc(&dt, (size_t)nframes * 24 * 4));
    CU(cudaMemsetAsync(dh, 0, ngt > 0 ? ngt : 1, c->stream));
    CU(cudaMemsetAsync(dt, 0, (size_t)(nframes > 0 ? nframes : 1) * 24 * 4, c->stream));
    if (ndet) {
        eval_match_kernel<<<cdiv(ndet, 128), 128, 0, c->cur>>>((const EvalBox*)dd, ndet, (const EvalBox*)dg, (const int32_t*)dof, nframes, c->d_simtab,
                                                               c->simtab_n, tol, (int32_t*)dst, (int32_t*)dm, (uint8_t*)dh, (int32_t*)dt);
        TRY(check_launch(c, "eval_match"));
    }
    if (ngt) {
        eval_tally_gt_kernel<<<cdiv(ngt, 128), 128, 0, c->cur>>>((const EvalBox*)dg, ngt, (const uint8_t*)dh, (int32_t*)dt);
        TRY(check_launch(c, "eval_tally_gt"));
    }
    if (ndet) { TRY(s.out(status, dst, (size_t)ndet * 4)); TRY(s.out(match, dm, (size_t)ndet * 4)); }
    if (nframes) TRY(s.out(tally, dt, (size_t)nframes * 24 * 4));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_match_iou(tsd_ctx* c, const int32_t* det, const int32_t* det_offsets, const int32_t* gt, const int32_t* gt_offsets, int nimages, double ovr,
                  uint8_t* tp, uint8_t* fp) {
    if (!c || nimages < 0 || !det_offsets || !gt_offsets) return fail(TSD_E_INVALID, "bad argument");
    const int ndet = det_offsets[nimages], ngt = gt_offsets[nimages];
    if (ndet < 0 || ngt < 0 || (ndet && (!det || !tp || !fp)) || (ngt && !gt)) return fail(TSD_E_INVALID, "bad argument");
    for (int i = 0; i < ndet; i++) if (det[5 * i + 4] < 0 || det[5 * i + 4] >= ndet) return fail(TSD_E_INVALID, "detection %d: list index out of range", i);
    CU(cudaSetDevice(c->device));
    if (nimages == 0 || ndet == 0) return TSD_OK;
    Stage s(c);
    void *dd, *ddo, *dg = nullptr, *dgo, *du, *dtp, *dfp;
    TRY(s.in(det, (size_t)ndet * 20, &dd));
    TRY(s.in(det_offsets, (size_t)(nimages + 1) * 4, &ddo));
    TRY(s.in(gt, (size_t)ngt * 20, &dg));
    TRY(s.in(gt_offsets, (size_t)(nimages + 1) * 4, &dgo));
    TRY(s.alloc(&du, (size_t)ngt));
    TRY(s.alloc(&dtp, (size_t)ndet));
    TRY(s.alloc(&dfp, (size_t)ndet));
    CU(cudaMemsetAsync(du, 0, ngt > 0 ? ngt : 1, c->stream));
    eval_iou_kernel<<<cdiv(nimages, 64), 64, 0, c->cur>>>((const EvalDt*)dd, (const int32_t*)ddo, (const EvalGt*)dg, (const int32_t*)dgo, nimages, ovr,
                                                          (uint8_t*)du, (uint8_t*)dtp, (uint8_t*)dfp);
    TRY(check_launch(c, "eval_iou"));
    TRY(s.out(tp, dtp, (size_t)ndet));
    TRY(s.out(fp, dfp, (size_t)ndet));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_bgr2hsv(tsd_ctx* c, const uint8_t* bgr, int64_t npx, uint8_t* hsv, int mem) {
    if (!c || npx < 0 || (npx && (!bgr || !hsv))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (npx == 0) return TSD_OK;
    Stage s(c);
    void *di = (void*)bgr, *dout = hsv;
    if (mem == TSD_MEM_HOST) { TRY(s.in(bgr, (size_t)npx * 3, &di)); TRY(s.alloc(&dout, (size_t)npx * 3)); }
    int grid = cdiv(npx, 256);
    if (grid > c->sm_count * 32) grid = c->sm_count * 32;
    bgr2hsv_kernel<<<grid, 256, 0, c->cur>>>((uint8_t*)di, npx, c->d_tab, (uint8_t*)dout);
    TRY(check_launch(c, "bgr2hsv"));
    if (mem == TSD_MEM_HOST) { TRY(s.out(hsv, dout, (size_t)npx * 3)); CU(cudaStreamSynchronize(c->stream)); }
    return TSD_OK;
}

int tsd_score_masks(tsd_ctx* c, const uint8_t* red, const uint8_t* blue, int n, int D, int32_t* scores, int32_t* id,
                    int32_t* hundredths, uint8_t* emit, int mem) {
    if (!c || n < 0 || (n && (!red || !blue || !id || !hundredths || !emit))) return fail(TSD_E_INVALID, "bad argument");
    if (!c->have_templates) return fail(TSD_E_STATE, "templates not set (tsd_set_templates)");
    if (D != c->tmpl_D) return fail(TSD_E_INVALID, "D=%d but templates are %dx%d", D, c->tmpl_D, c->tmpl_D);
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    const int npx = D * D;
    Stage s(c);
    void *dr = (void*)red, *db = (void*)blue, *ds = scores, *di = id, *dh = hundredths, *de = emit;
    if (mem == TSD_MEM_HOST) {
        TRY(s.in(red, (size_t)n * npx, &dr)); TRY(s.in(blue, (size_t)n * npx, &db));
        if (scores) TRY(s.alloc(&ds, (size_t)n * 12 * 4));
        TRY(s.alloc(&di, (size_t)n * 4)); TRY(s.alloc(&dh, (size_t)n * 4)); TRY(s.alloc(&de, (size_t)n));
    }
    k4_score_kernel<<<cdiv((int64_t)n * 32, 128), 128, 0, c->cur>>>((uint8_t*)dr, (uint8_t*)db, nullptr, n, npx, npx, c->d_tmpl,
                                                                        c->cfg.score_tol_hundredths, (int32_t*)ds, (int32_t*)di, (int32_t*)dh, (uint8_t*)de);
    TRY(check_launch(c, "k4_score"));
    if (mem == TSD_MEM_HOST) {
        if (scores) TRY(s.out(scores, ds, (size_t)n * 12 * 4));
        TRY(s.out(id, di, (size_t)n * 4)); TRY(s.out(hundredths, dh, (size_t)n * 4)); TRY(s.out(emit, de, (size_t)n));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

// K3 + K4 for a list of windows: detectionsMaskCorrelation (DET:229-245) per window, batched.  Host pointers.
int tsd_score(tsd_ctx* c, const uint8_t* windows, int n, int D, int32_t* id, int32_t* hundredths, uint8_t* emit, int mem) {
    if (!c || n < 0 || (n && (!windows || !id || !hundredths || !emit))) return fail(TSD_E_INVALID, "bad argument");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "tsd_score takes host pointers; use tsd_enqueue_frames for device-resident batches");
    if (!c->have_templates) return fail(TSD_E_STATE, "templates not set (tsd_set_templates)");
    if (D != c->tmpl_D) return fail(TSD_E_INVALID, "D=%d but templates are %dx%d", D, c->tmpl_D, c->tmpl_D);
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    const int npx = D * D;
    Stage s(c);
    void *dw, *dr, *db, *di, *dh, *de;
    TRY(s.in(windows, (size_t)n * npx * 3, &dw));
    TRY(s.alloc(&dr, (size_t)n * npx)); TRY(s.alloc(&db, (size_t)n * npx));
    TRY(s.alloc(&di, (size_t)n * 4)); TRY(s.alloc(&dh, (size_t)n * 4)); TRY(s.alloc(&de, (size_t)n));
    int grid = cdiv((int64_t)n * 32, 256);
    if (grid > c->sm_count * 8) grid = c->sm_count * 8;
    k3_masks_generic_kernel<<<grid, 256, 0, c->cur>>>((uint8_t*)dw, nullptr, nullptr, n, npx, npx * 3, c->d_tab, bounds_of(c->cfg), (uint8_t*)dr, (uint8_t*)db, npx, nullptr);
    TRY(check_launch(c, "k3_masks"));
    k4_score_kernel<<<cdiv((int64_t)n * 32, 128), 128, 0, c->cur>>>((uint8_t*)dr, (uint8_t*)db, nullptr, n, npx, npx, c->d_tmpl, c->cfg.score_tol_hundredths,
                                                                     nullptr, (int32_t*)di, (int32_t*)dh, (uint8_t*)de);
    TRY(check_launch(c, "k4_score"));
    TRY(s.out(id, di, (size_t)n * 4)); TRY(s.out(hundredths, dh, (size_t)n * 4)); TRY(s.out(emit, de, (size_t)n));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

int tsd_bgr2gray(tsd_ctx* c, const uint8_t* bgr, int64_t npx, uint8_t* gray, int mem) {
    if (!c || npx < 0 || npx > 0x7fffffffLL || (npx && (!bgr || !gray))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (npx == 0) return TSD_OK;
    Stage s(c);
    void *di = (void*)bgr, *dout = gray;
    if (mem == TSD_MEM_HOST) { TRY(s.in(bgr, (size_t)npx * 3, &di)); TRY(s.alloc(&dout, (size_t)npx)); }
    int grid = cdiv(npx, 256);
    if (grid > c->sm_count * 32) grid = c->sm_count * 32;
    k6_gray_kernel<<<grid, 256, 0, c->cur>>>((uint8_t*)di, nullptr, nullptr, 1, (int)npx, 0, (uint8_t*)dout);
    TRY(check_launch(c, "k6_gray"));
    if (mem == TSD_MEM_HOST) { TRY(s.out(gray, dout, (size_t)npx)); CU(cudaStreamSynchronize(c->stream)); }
    return TSD_OK;
}

int tsd_hog(tsd_ctx* c, const uint8_t* gray, int n, float* desc, int mem) {
    if (!c || n < 0 || (n && (!gray || !desc))) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    Stage s(c);
    void *dg = (void*)gray, *dd = desc;
    if (mem == TSD_MEM_HOST) { TRY(s.in(gray, (size_t)n * 1024, &dg)); TRY(s.alloc(&dd, (size_t)n * TSD_HOG_LEN * 4)); }
    {
        int grid = cdiv(n, kHogWarps);
        if (grid > c->sm_count * 8) grid = c->sm_count * 8;
        k7_hog_kernel<<<grid, kHogWarps * 32, 0, c->cur>>>((uint8_t*)dg, nullptr, n, c->hog, (float*)dd);
    }
    TRY(check_launch(c, "k7_hog"));
    if (mem == TSD_MEM_HOST) { TRY(s.out(desc, dd, (size_t)n * TSD_HOG_LEN * 4)); CU(cudaStreamSynchronize(c->stream)); }
    return TSD_OK;
}

static int dev_lda(tsd_ctx* c, const float* X, const int32_t* n_ptr, int n_max, double tol, double* logits, int32_t* labels) {
    int grid = cdiv((int64_t)n_max * 32, 256);
    if (grid > c->sm_count * 8) grid = c->sm_count * 8;
    k8_lda_kernel<<<grid, 256, (size_t)c->lda_nfeat * 6 * sizeof(double), c->cur>>>(X, n_ptr, n_max, c->lda_nfeat, c->d_ldaW, c->d_ldab, tol, logits, labels);
    return check_launch(c, "k8_lda");
}

int tsd_lda_predict(tsd_ctx* c, const float* X, int n, double tol, double* logits, int32_t* labels, int mem) {
    if (!c || n < 0 || (n && (!X || !labels))) return fail(TSD_E_INVALID, "bad argument");
    if (!c->d_ldaW) return fail(TSD_E_STATE, "LDA weights not set (tsd_set_lda)");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    Stage s(c);
    void *dx = (void*)X, *dl = logits, *dy = labels;
    if (mem == TSD_MEM_HOST) {
        TRY(s.in(X, (size_t)n * c->lda_nfeat * 4, &dx));
        if (logits) TRY(s.alloc(&dl, (size_t)n * 6 * 8));
        TRY(s.alloc(&dy, (size_t)n * 4));
    }
    TRY(dev_lda(c, (float*)dx, nullptr, n, tol, (double*)dl, (int32_t*)dy));
    if (mem == TSD_MEM_HOST) {
        if (logits) TRY(s.out(logits, dl, (size_t)n * 6 * 8));
        TRY(s.out(labels, dy, (size_t)n * 4));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

// K6 + K7 + K8 for a list of 32x32 BGR windows: BGR2GRAY (REC:388), HOG (REC:519), the six LDA probabilities and
// extractBestPredictions (REC:565-577,627-641).  Host pointers.
int tsd_recognize(tsd_ctx* c, const uint8_t* windows, int n, double tol, int32_t* labels, int mem) {
    if (!c || n < 0 || (n && (!windows || !labels))) return fail(TSD_E_INVALID, "bad argument");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "tsd_recognize takes host pointers; use tsd_enqueue_frames for device-resident batches");
    if (!c->d_ldaW || c->lda_nfeat != TSD_HOG_LEN) return fail(TSD_E_STATE, "324-feature LDA weights not set (tsd_set_lda)");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    Stage s(c);
    void *dw, *dg, *dh, *dl;
    TRY(s.in(windows, (size_t)n * 1024 * 3, &dw));
    TRY(s.alloc(&dg, (size_t)n * 1024)); TRY(s.alloc(&dh, (size_t)n * TSD_HOG_LEN * 4)); TRY(s.alloc(&dl, (size_t)n * 4));
    int grid = cdiv((int64_t)n * 1024, 256);
    if (grid > c->sm_count * 32) grid = c->sm_count * 32;
    k6_gray_kernel<<<grid, 256, 0, c->cur>>>((uint8_t*)dw, nullptr, nullptr, 1, n * 1024, 0, (uint8_t*)dg);
    TRY(check_launch(c, "k6_gray"));
    int hgrid = cdiv(n, kHogWarps);
    if (hgrid > c->sm_count * 8) hgrid = c->sm_count * 8;
    k7_hog_kernel<<<hgrid, kHogWarps * 32, 0, c->cur>>>((uint8_t*)dg, nullptr, n, c->hog, (float*)dh);
    TRY(check_launch(c, "k7_hog"));
    TRY(dev_lda(c, (float*)dh, nullptr, n, tol, nullptr, (int32_t*)dl));
    TRY(s.out(labels, dl, (size_t)n * 4));
    CU(cudaStreamSynchronize(c->stream));
    return TSD_OK;
}

// Evaluation entry point (north_star: "the batched LDA projection ... is evaluated for tensor cores (TF32) against FP32 FMA"):
// the same decision from TF32 tensor-core logits.  split = 1 (plain TF32) or 3 (3xTF32).  *ms (optional) receives the device time
// of the kernel alone (CUDA events).  NOT used by the chain: the product path is the f64 kernel (tsd_lda_predict).
int tsd_lda_predict_tf32(tsd_ctx* c, const float* X, int n, double tol, int split, float* logits, int32_t* labels, float* ms, int mem) {
    if (!c || n < 0 || (n && (!X || !labels)) || (split != 1 && split != 3)) return fail(TSD_E_INVALID, "bad argument");
    if (mem != TSD_MEM_HOST) return fail(TSD_E_INVALID, "host pointers only");
    if (!c->d_ldaW) return fail(TSD_E_STATE, "LDA weights not set (tsd_set_lda)");
    CU(cudaSetDevice(c->device));
    // the hi and lo TF32 tiles of W, [2][kpad][8] floats = 64 B per padded feature: up to 3 632 features on the B200
    const int kpad = (c->lda_nfeat + 7) & ~7;
    const size_t smem = (size_t)2 * kpad * 8 * sizeof(float);
    TRY(allow_dynamic_smem(c, split == 1 ? (const void*)k8_lda_tf32_kernel<1> : (const void*)k8_lda_tf32_kernel<3>, smem, "k8_lda_tf32"));
    if (n == 0) return TSD_OK;
    Stage s(c);
    void *dx, *dl, *dy;
    TRY(s.in(X, (size_t)n * c->lda_nfeat * 4, &dx));
    TRY(s.alloc(&dl, (size_t)n * 6 * 4));
    TRY(s.alloc(&dy, (size_t)n * 4));
    int grid = cdiv(cdiv(n, 16), 4);
    if (grid > c->sm_count * 8) grid = c->sm_count * 8;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    for (int rep = 0; rep < 2; rep++) {                      // first launch warms up, second is timed
        CU(cudaEventRecord(e0, c->cur));
        if (split == 1) k8_lda_tf32_kernel<1><<<grid, 128, smem, c->cur>>>((float*)dx, n, c->lda_nfeat, c->d_ldaW, c->d_ldab, tol, (float*)dl, (int32_t*)dy);
        else k8_lda_tf32_kernel<3><<<grid, 128, smem, c->cur>>>((float*)dx, n, c->lda_nfeat, c->d_ldaW, c->d_ldab, tol, (float*)dl, (int32_t*)dy);
        CU(cudaEventRecord(e1, c->cur));
        TRY(check_launch(c, "k8_lda_tf32"));
    }
    if (logits) TRY(s.out(logits, dl, (size_t)n * 6 * 4));
    TRY(s.out(labels, dy, (size_t)n * 4));
    CU(cudaStreamSynchronize(c->stream));
    if (ms) CU(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return TSD_OK;
}

int tsd_knn_predict(tsd_ctx* c, const float* X, int n, double* Z, int32_t* labels, int mem) {
    if (!c || n < 0 || (n && (!X || !labels))) return fail(TSD_E_INVALID, "bad argument");
    if (!c->d_Zt) return fail(TSD_E_STATE, "KNN model not set (tsd_set_knn)");
    CU(cudaSetDevice(c->device));
    if (n == 0) return TSD_OK;
    Stage s(c);
    void *dx = (void*)X, *dz = Z, *dy = labels;
    if (mem == TSD_MEM_HOST) {
        TRY(s.in(X, (size_t)n * c->knn_nfeat * 4, &dx));
        if (Z) TRY(s.alloc(&dz, (size_t)n * 6 * 8));
        TRY(s.alloc(&dy, (size_t)n * 4));
    }
    k8_knn_kernel<<<cdiv((int64_t)n * 32, 128), 128, 0, c->cur>>>((float*)dx, n, c->knn_nfeat, c->d_xbar, c->d_scal, c->d_Zt, c->d_yt,
                                                                      c->knn_ntrain, c->knn_k, (double*)dz, (int32_t*)dy);
    TRY(check_launch(c, "k8_knn"));
    if (mem == TSD_MEM_HOST) {
        if (Z) TRY(s.out(Z, dz, (size_t)n * 6 * 8));
        TRY(s.out(labels, dy, (size_t)n * 4));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

// ---- whole chain -------------------------------------------------------------------------------------------------
// One batch of frames through the whole chain on c->cur.  B.wo = first window slot of the batch in the per-window scratch,
// B.fo = first entry in the per-frame scratch arrays (nframes + 1 entries), B.nbcap = upper bound of the batch's windows;
// M = the batch's rows of the pair-class bit matrix.
static int enqueue_chain(tsd_ctx* c, int mode, const uint8_t* d_frames, int H, int W, int64_t row_stride, int64_t frame_stride,
                         const int32_t* d_boxes, const int32_t* d_box_offsets, int maxb, const tsd_ctx::Batch& B, uint32_t* M, int32_t* todo,
                         const uint8_t* host_src = nullptr /* page-locked host frames (device pointer): staged into d_frames (the mirror) after K1 */) {
    const int D = c->cfg.window, npx = D * D, nbytes = npx * 3, ws = win_stride(npx, 3), es = ent_stride(npx);
    const int ms = (npx + 15) & ~15, NW = (npx + 31) >> 5;     // mask byte stride (padded), mask words
    const int cf = B.nframes, nb = B.nbcap, fo = B.fo;
    const size_t cap = nb > 0 ? nb : 1, wo = B.wo;
    int32_t *cnt = (int32_t*)c->b_cnt.p + fo, *winoff = (int32_t*)c->b_winoff.p + fo, *survcnt = (int32_t*)c->b_survcnt.p + fo, *survoff = (int32_t*)c->b_survoff.p + fo;
    int32_t *detcnt = (int32_t*)c->b_detcnt.p + fo, *detoff = (int32_t*)c->b_detoff.p + fo;
    int32_t* coords = (int32_t*)c->b_coords.p + wo * 4;
    int32_t* winframe = (int32_t*)c->b_winframe.p + wo;
    uint8_t* windows = (uint8_t*)c->b_windows.p + wo * ws;
    uint32_t* entries = (uint32_t*)c->b_entries.p + wo * es;
    WinMeta* meta = (WinMeta*)c->b_meta.p + wo;
    float* energy = (float*)c->b_energy.p + wo * kEnergyRows;          // [25 energies + chunk boundaries][cap] block of this batch
    int32_t *list = (int32_t*)c->b_list.p + wo, *slots = (int32_t*)c->b_slots.p + wo, *id = (int32_t*)c->b_id.p + wo, *hund = (int32_t*)c->b_hund.p + wo;
    uint8_t *flags = (uint8_t*)c->b_flags.p + wo, *emit = (uint8_t*)c->b_emit.p + wo;
    DetRec* det = (DetRec*)c->b_det.p + wo;
    c->order_off = (size_t)fo;
    const int32_t* d_nwin = winoff + cf;
    // Two-slot overlap: consecutive batches run on two streams so that the latency-bound fold of one hides under the throughput-bound
    // front half (K1, K2, histograms, pair classes) of the next.  Left alone the two streams share the GPU evenly, drift into
    // phase and end up folding at the same time (3.24 ms per 4096-frame step against 2.6 ms of kernel work); making the front
    // half of a batch wait for the previous batch's keeps them a half period apart.
    const bool stagger = B.in_slot && c->stagger;
    if (stagger) TRY(ev_wait(c, c->ev_w1[B.sidx ^ 1]));
    mark(c, "start");
    // K1: candidate loop of MSERTrafficSignDetector (DET:116-120)
    TRY(dev_windows_index(c, d_boxes, d_box_offsets, cf, H, W, c->cfg.enlarge, cnt, winoff, coords, winframe));
    mark(c, "k1_expand_filter");
    if (host_src) {                                          // every 32-byte sector the ROIs touch crosses PCIe once, into the mirror
        const int wpr = (cdiv((int64_t)W * 3, 32) + 31) / 32;
        const int64_t nwords = (int64_t)cf * H * wpr;
        uint32_t* stagemap = (uint32_t*)c->b_stagemap[B.sidx].p;
        CU(cudaMemsetAsync(stagemap, 0, (size_t)nwords * 4, c->cur));
        if (nb > 0) {
            stage_mark_kernel<<<cdiv((int64_t)nb * 32, 128), 128, 0, c->cur>>>((const int4*)coords, winframe, d_nwin, nb, H, W, D, wpr, c->stage_gran, stagemap);
            TRY(check_launch(c, "stage_mark"));
            int g = cdiv(nwords, 256);
            if (g > c->sm_count * c->stage_ctas) g = c->sm_count * c->stage_ctas;
            stage_copy_kernel<<<g, 256, 0, c->cur>>>(host_src, row_stride, frame_stride, H, W * 3, wpr, nwords, stagemap,
                                                     (uint8_t*)d_frames, c->d_staged);
            TRY(check_launch(c, "stage_copy"));
        }
        // PCIe is the serial resource of a host-staged batch: the next batch's staging may start as soon as this one's has ended
        if (stagger) TRY(ev_record(c, c->ev_w1[B.sidx]));
        mark(c, "stage_h2d");
    }
    // K2 (DET:123-124)
    TRY(dev_crop_resize(c, d_frames, H, W, row_stride, frame_stride, 3, coords, winframe, d_nwin, nb, D, windows, ws, cf));
    mark(c, "k2_crop_resize");
    // K5 (DET:127-129)
    TRY(dev_hist(c, windows, d_nwin, nb, npx, ws, entries, meta, energy, (int64_t)cap));
    mark(c, "k5_hist");
    TRY(dev_fold(c, windows, ws, coords, entries, meta, winoff, cf, npx, 1, 1, c->cfg.hist_tol, c->cfg.coord_tol,
                 list, flags, survcnt, maxb, M, todo, energy, (int64_t)cap, survoff, (stagger && !host_src) ? c->ev_w1[B.sidx] : nullptr));
    k5_gather_kernel<<<cf, 32, 0, c->cur>>>(windows, (int4*)coords, winoff, list, survoff, cf, nbytes, ws, nullptr, nullptr, slots);
    TRY(check_launch(c, "k5_gather"));
    mark(c, "k5_fold");
    const int32_t* d_nsurv = survoff + cf;
    if (mode == TSD_RUN_DETECT) {
        // K3 + K4 (DET:708-716)
        uint8_t *red = (uint8_t*)c->b_red.p + wo * ms, *blue = (uint8_t*)c->b_blue.p + wo * ms;
        uint32_t* bits = (uint32_t*)c->b_bits.p + wo * 2 * NW;
        int grid = cdiv((int64_t)cap * 32, 256);
        if (grid > c->sm_count * TSD_K3_GRID) grid = c->sm_count * TSD_K3_GRID;
        // K4 reads the bit-packed masks at NW = 20 / 32 words (D = 25, 29..32) and the byte masks at every other D.  K3 v3 writes the
        // byte masks only when K4 reads them or TSD_KEEP_MASKS=1 asks for them (the generic kernel always writes both)
        const bool k4_bits = NW == 20 || NW == 32;
        const bool want_bytes = c->keep_masks || !k4_bits;
        if (ws <= 4 * 32 * 16)
            k3_masks_v3_kernel<4><<<grid, 256, 0, c->cur>>>(windows, slots, d_nsurv, nb, npx, ws, c->d_tab, c->d_mlut, want_bytes ? red : nullptr,
                                                            want_bytes ? blue : nullptr, ms, bits);
        else
            k3_masks_generic_kernel<<<grid, 256, 0, c->cur>>>(windows, slots, d_nsurv, nb, npx, ws, c->d_tab, bounds_of(c->cfg), red, blue, ms, bits);
        TRY(check_launch(c, "k3_masks"));
        mark(c, "k3_masks");
        if (NW == 20)
            k4_score_bits_kernel<20><<<cdiv(cap, 128), 128, 0, c->cur>>>(bits, d_nsurv, nb, c->d_tmpl, c->cfg.score_tol_hundredths, id, hund, emit);
        else if (NW == 32)
            k4_score_bits_kernel<32><<<cdiv(cap, 128), 128, 0, c->cur>>>(bits, d_nsurv, nb, c->d_tmpl, c->cfg.score_tol_hundredths, id, hund, emit);
        else
            k4_score_kernel<<<cdiv((int64_t)cap * 32, 128), 128, 0, c->cur>>>(red, blue, d_nsurv, nb, npx, ms, c->d_tmpl, c->cfg.score_tol_hundredths, nullptr, id, hund, emit);
        TRY(check_launch(c, "k4_score"));
        mark(c, "k4_score");
    } else {
        uint8_t* gray = (uint8_t*)c->b_gray.p + wo * npx;
        float* hog = (float*)c->b_hog.p + wo * TSD_HOG_LEN;
        int grid = cdiv((int64_t)cap * npx, 256);
        if (grid > c->sm_count * 16) grid = c->sm_count * 16;
        k6_gray_kernel<<<grid, 256, 0, c->cur>>>(windows, slots, d_nsurv, nb, npx, ws, gray);
        TRY(check_launch(c, "k6_gray"));
        mark(c, "k6_gray");
        {
            int hgrid = cdiv(cap, kHogWarps);
            if (hgrid > c->sm_count * 8) hgrid = c->sm_count * 8;
            k7_hog_kernel<<<hgrid, kHogWarps * 32, 0, c->cur>>>(gray, d_nsurv, nb, c->hog, hog);
        }
        TRY(check_launch(c, "k7_hog"));
        mark(c, "k7_hog");
        TRY(dev_lda(c, hog, d_nsurv, nb, c->cfg.proba_tol, nullptr, id));
        mark(c, "k8_lda");
        // a survivor becomes a record when the classifier says "sign" (label != 0); no score in this flavour
        CU(cudaMemsetAsync(hund, 0, cap * 4, c->cur));
        label_emit_kernel<<<cdiv(cap, 256), 256, 0, c->cur>>>(id, d_nsurv, nb, emit);
        TRY(check_launch(c, "label_emit"));
    }
    det_count_kernel<<<cdiv((int64_t)cf * 32, 128), 128, 0, c->cur>>>(emit, survoff, cf, detcnt, detoff, c->d_tickets + c->ticket_base + 2);
    TRY(check_launch(c, "det_count"));
    det_write_kernel<<<cdiv((int64_t)cf * 32, 128), 128, 0, c->cur>>>(emit, id, hund, (int4*)coords, slots, survoff, detoff, cf, (int)cap, det,
                                                                        winoff + cf, survoff + cf, (int32_t*)c->b_summary.p + 4 * B.sidx);
    TRY(check_launch(c, "det_write"));
    mark(c, "detections");
    return TSD_OK;
}

// One batch through the chain on c->cur: eagerly the first time a batch shape is seen, captured into a CUDA graph the second time,
// replayed from then on (at most 8 graphs are kept, least recently used goes first).
static int run_chain(tsd_ctx* c, int mode, const uint8_t* d_frames, int H, int W, int64_t row_stride, int64_t frame_stride,
                     const int32_t* d_boxes, const int32_t* d_box_offsets, int maxb, const tsd_ctx::Batch& B, uint32_t* M, int32_t* todo,
                     const uint8_t* host_src) {
    if (!c->use_graph || c->profiling)
        return enqueue_chain(c, mode, d_frames, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, maxb, B, M, todo, host_src);
    const std::vector<uint64_t> key = {(uint64_t)mode, (uint64_t)(uintptr_t)d_frames, (uint64_t)B.nframes, (uint64_t)H, (uint64_t)W, (uint64_t)row_stride,
                                       (uint64_t)frame_stride, (uint64_t)(uintptr_t)d_boxes, (uint64_t)(uintptr_t)d_box_offsets, (uint64_t)B.nbcap, (uint64_t)maxb,
                                       (uint64_t)B.wo, (uint64_t)B.fo, (uint64_t)B.sidx, (uint64_t)(uintptr_t)M, (uint64_t)(uintptr_t)todo,
                                       (uint64_t)c->ticket_base, c->gen, (uint64_t)c->keep_masks, (uint64_t)c->use_gram, (uint64_t)(uintptr_t)host_src, (uint64_t)c->fold_cta_cost, (uint64_t)c->fold_per_sm_cap, (uint64_t)c->k2_grid, (uint64_t)c->stagger, (uint64_t)c->stage_ctas, (uint64_t)c->stage_gran, (uint64_t)c->k2_tma};
    c->graph_clock++;
    for (auto& g : c->graphs)
        if (g.key == key) {
            CU(cudaGraphLaunch(g.exec, c->cur));
            g.stamp = c->graph_clock;
            c->launches += g.launches;
            return TSD_OK;
        }
    if (c->seen_key != key) {                                // first sighting: run it eagerly (one-off calls never pay for an instantiation)
        c->seen_key = key;
        return enqueue_chain(c, mode, d_frames, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, maxb, B, M, todo, host_src);
    }
    c->seen_key.clear();
    const int64_t l0 = c->launches;
    CU(cudaStreamBeginCapture(c->cur, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue_chain(c, mode, d_frames, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, maxb, B, M, todo, host_src);
    cudaGraph_t graph = nullptr;
    const cudaError_t ee = cudaStreamEndCapture(c->cur, &graph);
    if (rc != TSD_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (ee != cudaSuccess) return fail(TSD_E_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ee));
    tsd_ctx::GraphEntry g;
    g.key = key; g.launches = c->launches - l0; g.stamp = c->graph_clock;
    const cudaError_t ei = cudaGraphInstantiate(&g.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) return fail(TSD_E_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ei));
    if (c->graphs.size() >= 8) {
        size_t lru = 0;
        for (size_t i = 1; i < c->graphs.size(); i++) if (c->graphs[i].stamp < c->graphs[lru].stamp) lru = i;
        cudaGraphExecDestroy(c->graphs[lru].exec);
        c->graphs.erase(c->graphs.begin() + lru);
    }
    c->graphs.push_back(g);
    CU(cudaGraphLaunch(g.exec, c->cur));
    return TSD_OK;
}

// host_src != NULL: d_frames is ignored, the frames are page-locked host memory (host_src = their device pointer) and are staged
// ROI sector by ROI sector into the context's mirror, which the chain then reads.
static int enqueue_impl(tsd_ctx* c, int mode, const uint8_t* d_frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride,
                        const int32_t* d_boxes, const int32_t* d_box_offsets, int nb, int max_boxes_per_frame, const uint8_t* host_src) {
    if (host_src) d_frames = host_src;                       // (argument checks below)
    if (!c || !d_frames || !d_box_offsets || nframes < 1 || nb < 0 || H < 1 || W < 1) return fail(TSD_E_INVALID, "bad argument");
    if (mode != TSD_RUN_DETECT && mode != TSD_RUN_RECOGNIZE) return fail(TSD_E_INVALID, "bad mode %d", mode);
    if (row_stride < (int64_t)W * 3 || frame_stride < row_stride * (H - 1) + (int64_t)W * 3) return fail(TSD_E_INVALID, "bad strides");
    const int D = c->cfg.window, npx = D * D, ws = win_stride(npx, 3), es = ent_stride(npx);
    const int ms = (npx + 15) & ~15, NW = (npx + 31) >> 5;
    if (mode == TSD_RUN_DETECT && (!c->have_templates || c->tmpl_D != D)) return fail(TSD_E_STATE, "templates not set for D=%d", D);
    if (mode == TSD_RUN_RECOGNIZE && (!c->d_ldaW || D != 32 || c->lda_nfeat != TSD_HOG_LEN)) return fail(TSD_E_STATE, "recognition needs D=32 and 324-feature LDA weights");
    CU(cudaSetDevice(c->device));
    if (max_boxes_per_frame <= 0) {                          // not given: one small D2H of the CSR offsets (synchronises)
        std::vector<int32_t> ho(nframes + 1);
        CU(cudaMemcpyAsync(ho.data(), d_box_offsets, (size_t)(nframes + 1) * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        for (int f = 0; f < nframes; f++) max_boxes_per_frame = ho[f + 1] - ho[f] > max_boxes_per_frame ? ho[f + 1] - ho[f] : max_boxes_per_frame;
    }
    const int RW = pair_row_words(max_boxes_per_frame);
    c->prev = c->last;                                       // (tsd_fetch_previous: valid only while both batches sit in slots)
    if (!c->prev.in_slot) c->prev.valid = false;
    c->last = tsd_ctx::Batch();
    tsd_ctx::Batch B;
    B.nframes = nframes; B.nbcap = nb; B.nboxes = nb;
    const size_t need_w = (((size_t)(nb > 0 ? nb : 1) + 3) & ~(size_t)3);
    const size_t need_todo = 2 * todo_capacity(nframes, max_boxes_per_frame);      // work lists of k5_pairs and k5_gram_big
    size_t cap = need_w, fcap = (size_t)nframes + 2, mwords = need_w * 2 * RW, m_off = 0, todo_words = need_todo, todo_off = 0;
    const bool ov = c->overlap && c->profiling != 1;
    if (ov) {                                                // this batch lives in slot `slot` of doubled scratch buffers
        c->slot ^= 1;
        const size_t sw = (need_w + 63) & ~(size_t)63, sf = ((size_t)nframes + 2 + 63) & ~(size_t)63;
        if (sw > c->slot_cap || sf > c->slot_fcap || RW > c->slot_rw || need_todo > c->slot_todo) {
            // The slot layout changes (slot 1 starts at slot_cap windows, slot_fcap frames, slot_cap * 2 * slot_rw pair-class
            // words): nothing may be in flight in either slot.  All three are sticky maxima, so a batch never reaches into the
            // other slot whatever its own RW is.
            c->prev.valid = false;
            TRY(join_pending(c));
            CU(cudaStreamSynchronize(c->stream));
            if (sw > c->slot_cap) c->slot_cap = sw;
            if (sf > c->slot_fcap) c->slot_fcap = sf;
            if (RW > c->slot_rw) c->slot_rw = RW;
            if (need_todo > c->slot_todo) c->slot_todo = need_todo;
            c->gen++;
        }
        B.wo = (size_t)c->slot * c->slot_cap;
        B.fo = (int)((size_t)c->slot * c->slot_fcap);
        B.sidx = c->slot; B.in_slot = true;
        cap = 2 * c->slot_cap; fcap = 2 * c->slot_fcap;
        mwords = 2 * c->slot_cap * 2 * (size_t)c->slot_rw;
        m_off = (size_t)c->slot * c->slot_cap * 2 * (size_t)c->slot_rw;
        todo_words = 2 * c->slot_todo; todo_off = (size_t)c->slot * c->slot_todo;
    } else {
        TRY(join_pending(c));
        c->prev.valid = false;
    }
    TRY(ensure(c, c->b_cnt, fcap * 4));
    TRY(ensure(c, c->b_winoff, fcap * 4));
    TRY(ensure(c, c->b_survcnt, fcap * 4));
    TRY(ensure(c, c->b_survoff, fcap * 4));
    TRY(ensure(c, c->b_detcnt, fcap * 4));
    TRY(ensure(c, c->b_detoff, fcap * 4));
    TRY(ensure(c, c->b_summary, 2 * 16));
    TRY(ensure(c, c->b_order, (2 * fcap + 4) * 4));
    TRY(ensure(c, c->b_gramdone, todo_words * 4));
    TRY(ensure(c, c->b_coords, cap * 16));
    TRY(ensure(c, c->b_winframe, cap * 4));
    TRY(ensure(c, c->b_windows, cap * ws));
    TRY(ensure(c, c->b_entries, cap * es * 4));
    TRY(ensure(c, c->b_meta, cap * sizeof(WinMeta)));
    TRY(ensure(c, c->b_energy, cap * kEnergyRows * 4));
    TRY(ensure(c, c->b_list, cap * 4));
    TRY(ensure(c, c->b_flags, cap));
    TRY(ensure(c, c->b_slots, cap * 4));
    TRY(ensure(c, c->b_id, cap * 4));
    TRY(ensure(c, c->b_hund, cap * 4));
    TRY(ensure(c, c->b_emit, cap));
    TRY(ensure(c, c->b_det, cap * sizeof(DetRec)));
    if (mode == TSD_RUN_DETECT) {
        TRY(ensure(c, c->b_red, cap * ms));
        TRY(ensure(c, c->b_blue, cap * ms));
        TRY(ensure(c, c->b_bits, cap * 2 * NW * 4));
    } else {
        TRY(ensure(c, c->b_gray, cap * npx));
        TRY(ensure(c, c->b_hog, cap * TSD_HOG_LEN * 4));
    }
    TRY(ensure(c, c->b_pairs, mwords * sizeof(uint32_t)));
    if (host_src) {
        const int wpr = (cdiv((int64_t)W * 3, 32) + 31) / 32;
        const int ms_slot = ov ? c->slot : 0;                // (a grow frees + reallocates: cudaFree waits for the device)
        TRY(ensure(c, c->b_mirror[ms_slot], (size_t)frame_stride * (nframes - 1) + (size_t)row_stride * (H - 1) + (size_t)W * 3 + 64));
        TRY(ensure(c, c->b_stagemap[ms_slot], (size_t)nframes * H * wpr * 4));
        d_frames = (const uint8_t*)c->b_mirror[ms_slot].p;
    }
    uint32_t* M = (uint32_t*)c->b_pairs.p + m_off;
    int32_t* todo = (int32_t*)c->b_gramdone.p + todo_off;
    int rc = TSD_OK;
    if (ov) {
        const int sl = c->slot;
        CU(cudaEventRecord(c->ev_slot_fork[sl], c->stream));
        CU(cudaStreamWaitEvent(c->os[sl], c->ev_slot_fork[sl], 0));
        TRY(join_pending(c));                                // the PREVIOUS batch: the context's stream waits for it only now, after this batch's fork
        c->cur = c->os[sl];
        c->ticket_base = 8 * sl;
        rc = run_chain(c, mode, d_frames, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, max_boxes_per_frame, B, M, todo, host_src);
        CU(cudaEventRecord(c->ev_join[sl], c->os[sl]));
        c->pending_join = sl;
    } else {
        c->cur = c->stream;
        rc = run_chain(c, mode, d_frames, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, max_boxes_per_frame, B, M, todo, host_src);
    }
    c->cur = c->stream;
    c->ticket_base = 16;
    if (rc != TSD_OK) { c->prev.valid = false; return rc; }
    B.valid = true;
    c->last = B;
    c->last_mode = mode;
    if (!ov) c->prev.valid = false;
    return TSD_OK;
}

int tsd_enqueue_frames(tsd_ctx* c, int mode, const uint8_t* d_frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride,
                       const int32_t* d_boxes, const int32_t* d_box_offsets, int nb, int max_boxes_per_frame) {
    return enqueue_impl(c, mode, d_frames, nframes, H, W, row_stride, frame_stride, d_boxes, d_box_offsets, nb, max_boxes_per_frame, nullptr);
}

// Bytes the ROI staging of tsd_detect_frames (page-locked host frames) has copied over PCIe since process start / the last reset:
// 32 bytes per distinct sector a batch's candidate ROIs touch.  Synchronises.
int tsd_stat_staged_bytes(tsd_ctx* c, int64_t* total, int reset) {
    if (!c || !total) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    unsigned long long h = 0;
    CU(cudaMemcpy(&h, c->d_staged, 8, cudaMemcpyDeviceToHost));
    if (reset) CU(cudaMemset(c->d_staged, 0, 8));
    *total = (int64_t)h;
    return TSD_OK;
}

// Sum of the sparse-histogram lengths (non-zero bins) of the windows of the last tsd_enqueue_frames call: bench.py uses it
// for the algorithmic bytes of k5_pairs (every window's sparse histogram is read at least once).  Synchronises.
__global__ void sum_nnz_kernel(const WinMeta* __restrict__ meta, const int32_t* __restrict__ n_ptr, unsigned long long* __restrict__ out) {
    const int n = *n_ptr;
    unsigned long long acc = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) acc += (unsigned)meta[i].nnz;
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

int tsd_stat_hist_entries(tsd_ctx* c, int64_t* total) {
    if (!c || !total) return fail(TSD_E_INVALID, "bad argument");
    if (!c->last.valid) return fail(TSD_E_STATE, "nothing enqueued");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    unsigned long long* d = nullptr;
    CU(cudaMallocAsync((void**)&d, 8, c->stream));
    CU(cudaMemsetAsync(d, 0, 8, c->stream));
    sum_nnz_kernel<<<64, 256, 0, c->stream>>>((const WinMeta*)c->b_meta.p + c->last.wo, (const int32_t*)c->b_winoff.p + c->last.fo + c->last.nframes, d);
    unsigned long long h = 0;
    CU(cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaFreeAsync(d, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *total = (int64_t)h;
    return TSD_OK;
}

// Pairs (over the life of the process, all contexts of this device) that were decided by the exact f64 evaluation because their
// integer-dot classification came within 2e-6 of a threshold.  reset != 0 zeroes the counter after reading.  Synchronises.
int tsd_stat_unsure_pairs(tsd_ctx* c, int64_t* total, int reset) {
    if (!c || !total) return fail(TSD_E_INVALID, "bad argument");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    CU(cudaStreamSynchronize(c->stream));
    unsigned long long h = 0;
    CU(cudaMemcpyFromSymbol(&h, g_unsure_pairs, sizeof h));
    if (reset) { const unsigned long long z = 0; CU(cudaMemcpyToSymbol(g_unsure_pairs, &z, sizeof z)); }
    *total = (int64_t)h;
    return TSD_OK;
}

static int fetch_impl(tsd_ctx* c, const tsd_ctx::Batch& B, tsd_detection* det, int det_cap, int32_t* ndet, int32_t* counts) {
    static_assert(sizeof(tsd_detection) == sizeof(DetRec), "record layout");
    int32_t h[4] = {0, 0, 0, 0};                             // {windows, survivors, detections, -} written by det_write
    CU(cudaMemcpyAsync(h, (int32_t*)c->b_summary.p + 4 * B.sidx, 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (counts) { counts[0] = B.nboxes; counts[1] = h[0]; counts[2] = h[1]; counts[3] = h[2]; }
    *ndet = h[2];
    if (h[2] > det_cap) return fail(TSD_E_NOMEM, "det_cap %d < %d detections", det_cap, h[2]);
    if (h[2]) {
        if (!det) return fail(TSD_E_INVALID, "det is NULL");
        CU(cudaMemcpyAsync(det, (DetRec*)c->b_det.p + B.wo, (size_t)h[2] * sizeof(DetRec), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    return TSD_OK;
}

int tsd_fetch_detections(tsd_ctx* c, tsd_detection* det, int det_cap, int32_t* ndet, int32_t* counts) {
    if (!c || !ndet || det_cap < 0) return fail(TSD_E_INVALID, "bad argument");
    if (!c->last.valid) return fail(TSD_E_STATE, "nothing enqueued");
    CU(cudaSetDevice(c->device));
    TRY(join_pending(c));
    return fetch_impl(c, c->last, det, det_cap, ndet, counts);
}

// The batch enqueued BEFORE the last one (overlap mode): the context's stream already waits for it (the last tsd_enqueue_frames
// joined it after forking its own batch) but not for the last batch, which keeps running while these records are read.
int tsd_fetch_previous(tsd_ctx* c, tsd_detection* det, int det_cap, int32_t* ndet, int32_t* counts) {
    if (!c || !ndet || det_cap < 0) return fail(TSD_E_INVALID, "bad argument");
    if (!c->prev.valid || c->pending_join < 0)
        return fail(TSD_E_STATE, "no previous batch to fetch (needs two consecutive tsd_enqueue_frames calls in overlap mode, nothing in between)");
    CU(cudaSetDevice(c->device));
    const int rc = fetch_impl(c, c->prev, det, det_cap, ndet, counts);
    c->prev.valid = false;
    return rc;
}

int tsd_detect_frames(tsd_ctx* c, int mode, const uint8_t* frames, int nframes, int H, int W, int64_t row_stride, int64_t frame_stride,
                      const int32_t* boxes, const int32_t* box_offsets, tsd_detection* det, int det_cap, int32_t* ndet, int32_t* counts, int mem) {
    if (!c || !frames || !box_offsets || nframes < 1 || H < 1 || W < 1) return fail(TSD_E_INVALID, "bad argument");
    if (row_stride < (int64_t)W * 3 || frame_stride < row_stride * (H - 1) + (int64_t)W * 3) return fail(TSD_E_INVALID, "bad strides");
    CU(cudaSetDevice(c->device));
    if (mem == TSD_MEM_DEVICE) {
        int32_t nb = 0;
        CU(cudaMemcpyAsync(&nb, box_offsets + nframes, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        TRY(tsd_enqueue_frames(c, mode, frames, nframes, H, W, row_stride, frame_stride, boxes, box_offsets, nb, 0));
        return tsd_fetch_detections(c, det, det_cap, ndet, counts);
    }
    const int nb = box_offsets[nframes];
    if (nb < 0 || (nb && !boxes)) return fail(TSD_E_INVALID, "boxes is NULL");
    if (!ndet || det_cap < 0) return fail(TSD_E_INVALID, "bad argument");
    for (int f = 0; f < nframes; f++) if (box_offsets[f + 1] < box_offsets[f]) return fail(TSD_E_INVALID, "box_offsets must not decrease (frame %d)", f);
    // boxes + offsets: one small upload
    TRY(join_pending(c));
    TRY(ensure(c, c->b_hboxes, (size_t)(nb > 0 ? nb : 1) * 16));
    TRY(ensure(c, c->b_hoff, (size_t)(nframes + 1) * 4));
    if (nb) CU(cudaMemcpyAsync(c->b_hboxes.p, boxes, (size_t)nb * 16, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->b_hoff.p, box_offsets, (size_t)(nframes + 1) * 4, cudaMemcpyHostToDevice, c->stream));
    const int32_t* d_boxes = (const int32_t*)c->b_hboxes.p;
    const int32_t* d_off = (const int32_t*)c->b_hoff.p;
    int32_t tot[4] = {0, 0, 0, 0};
    int nd_total = 0;
    auto run_chunk = [&](const uint8_t* d_frames, int f0, int cf, const uint8_t* host_src = nullptr) -> int {
        int max_n = 0;
        for (int f = f0; f < f0 + cf; f++) max_n = box_offsets[f + 1] - box_offsets[f] > max_n ? box_offsets[f + 1] - box_offsets[f] : max_n;
        // offsets stay absolute: the kernels index `boxes` with them, so the base pointer is the whole box array
        return enqueue_impl(c, mode, d_frames, cf, H, W, row_stride, frame_stride, d_boxes, d_off + f0, box_offsets[f0 + cf] - box_offsets[f0], max_n > 0 ? max_n : 1, host_src);
    };
    auto fetch_chunk = [&](int f0) -> int {
        int32_t nd = 0, cnt[4];
        const int room = det_cap - nd_total;
        int rc = tsd_fetch_detections(c, det ? det + nd_total : nullptr, room > 0 ? room : 0, &nd, cnt);
        if (rc == TSD_E_NOMEM) { nd_total += nd; for (int i = 0; i < 4; i++) tot[i] += cnt[i]; return rc; }
        TRY(rc);
        for (int i = 0; i < nd; i++) det[nd_total + i].frame += f0;
        nd_total += nd;
        for (int i = 0; i < 4; i++) tot[i] += cnt[i];
        return TSD_OK;
    };
    int rc_all = TSD_OK;
    if (c->zero_copy) {
        // Page-locked (pinned / cudaHostRegister'ed) host frames are read IN PLACE: only the bytes of the candidate ROIs cross PCIe
        // (~0.3 MB of a 3.26 MB frame at 200 candidates).  Default: the mark + copy kernels bring every touched 32-byte sector over
        // once, coalesced, into a device mirror (needs 16-byte aligned frames and strides); TSD_STAGE=0: K2 gathers from host memory.
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
            const uint8_t* hp = (const uint8_t*)at.devicePointer;
            const bool stage = c->stage_rois && ((uintptr_t)hp % 16 == 0) && row_stride % 16 == 0 && frame_stride % 16 == 0 && ((int64_t)W * 3) % 16 == 0;
            const int SC = c->stage_chunk;
            if (stage && c->overlap && c->profiling != 1 && SC > 0 && nframes >= 2 * SC) {
                // Chunks of SC frames through the two scratch slots: the staging copy of chunk k+1 (PCIe-bound, a few resident warps)
                // runs beside the chain of chunk k; the records of chunk k are read once chunk k+1 is enqueued.
                int rc_chunks = TSD_OK, f_prev = -1;
                const int nchunks = nframes / SC < 4 ? nframes / SC : 4;     // (at most 4: every chunk shape is one cached CUDA graph)
                const int CFc = (nframes + nchunks - 1) / nchunks;
                for (int f0 = 0; f0 < nframes; f0 += CFc) {
                    const int cf = nframes - f0 < CFc ? nframes - f0 : CFc;
                    TRY(run_chunk(nullptr, f0, cf, hp + (size_t)f0 * frame_stride));
                    if (f_prev >= 0) {
                        int32_t nd = 0, cnt[4];
                        const int room = det_cap - nd_total;
                        const int rc = tsd_fetch_previous(c, det ? det + nd_total : nullptr, room > 0 ? room : 0, &nd, cnt);
                        if (rc != TSD_OK && rc != TSD_E_NOMEM) return rc;
                        if (rc == TSD_E_NOMEM) rc_chunks = rc;
                        else for (int i = 0; i < nd; i++) det[nd_total + i].frame += f_prev;
                        nd_total += nd;
                        for (int i = 0; i < 4; i++) tot[i] += cnt[i];
                    }
                    f_prev = f0;
                }
                const int rc = fetch_chunk(f_prev);
                *ndet = nd_total;
                if (counts) for (int i = 0; i < 4; i++) counts[i] = tot[i];
                if (rc != TSD_OK) return rc;
                if (rc_chunks != TSD_OK) return fail(TSD_E_NOMEM, "det_cap %d < %d detections", det_cap, nd_total);
                return TSD_OK;
            }
            TRY(stage ? run_chunk(nullptr, 0, nframes, hp) : run_chunk(hp, 0, nframes));
            const int rc = fetch_chunk(0);
            *ndet = nd_total;
            if (counts) for (int i = 0; i < 4; i++) counts[i] = tot[i];
            return rc;
        }
        cudaGetLastError();
    }
    // pageable frames: chunked, double-buffered whole-frame copies; the H2D copy of chunk k+1 (copy stream) overlaps the chain of chunk k
    const int CF = c->chunk_frames < nframes ? c->chunk_frames : nframes;
    const int nchunks = (nframes + CF - 1) / CF;
    const size_t frame_bytes = (size_t)row_stride * (H - 1) + (size_t)W * 3;
    auto chunk_bytes = [&](int cf) { return ((size_t)frame_stride * (cf - 1) + frame_bytes + 15) & ~(size_t)15; };
    for (int i = 0; i < (nchunks > 1 ? 2 : 1); i++) TRY(ensure(c, c->b_stage[i], chunk_bytes(CF)));
    auto issue_copy = [&](int k) -> int {
        const int slot = k & 1, f0 = k * CF, cf = nframes - f0 < CF ? nframes - f0 : CF;
        if (k >= 2) CU(cudaStreamWaitEvent(c->copy_stream, c->ev_consumed[slot], 0));
        CU(cudaMemcpyAsync(c->b_stage[slot].p, frames + (size_t)f0 * frame_stride, (size_t)frame_stride * (cf - 1) + frame_bytes, cudaMemcpyHostToDevice, c->copy_stream));
        CU(cudaEventRecord(c->ev_copied[slot], c->copy_stream));
        return TSD_OK;
    };
    TRY(issue_copy(0));
    for (int k = 0; k < nchunks; k++) {
        const int slot = k & 1, f0 = k * CF, cf = nframes - f0 < CF ? nframes - f0 : CF;
        if (k + 1 < nchunks) TRY(issue_copy(k + 1));
        CU(cudaStreamWaitEvent(c->stream, c->ev_copied[slot], 0));
        TRY(run_chunk((const uint8_t*)c->b_stage[slot].p, f0, cf));
        int rc = fetch_chunk(f0);                            // joins + synchronises the chunk's streams; the next copy is already in flight
        CU(cudaEventRecord(c->ev_consumed[slot], c->stream)); // (after the join: the batch ran on an internal stream)
        if (rc == TSD_E_NOMEM) rc_all = rc; else TRY(rc);
    }
    CU(cudaStreamSynchronize(c->copy_stream));
    *ndet = nd_total;
    if (counts) for (int i = 0; i < 4; i++) counts[i] = tot[i];
    if (rc_all != TSD_OK) return fail(TSD_E_NOMEM, "det_cap %d < %d detections", det_cap, nd_total);
    return TSD_OK;
}

}  // extern "C"

