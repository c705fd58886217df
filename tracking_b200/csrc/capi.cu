// C ABI of libbgsb200: background-subtraction contexts (include/bgsb200.h).
// Host-side bookkeeping only -- frame counters, warm-up rules, learning-rate schedule, buffer
// ownership -- mirroring what each reference plugin keeps in its members:
//   FrameDifferenceBGS   img_input_prev                     package_bgs/FrameDifferenceBGS.h
//   WeightedMovingVariance img_input_prev_1/2               package_bgs/WeightedMovingVarianceBGS.h
//   AdaptiveBackgroundLearning img_background               package_bgs/AdaptiveBackgroundLearning.h
//   MixtureOfGaussianV2BGS  cv::BackgroundSubtractorMOG2 mog package_bgs/MixtureOfGaussianV2BGS.h:30
#include <stdarg.h>
#include <string.h>
#include <algorithm>

#include <chrono>
#include <cstdlib>
#include <nvtx3/nvToolsExt.h>
#include "common.cuh"
#include "kernels.h"

namespace bgsb {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

}  // namespace bgsb

using namespace bgsb;

struct bgsb_ctx {
    int algo = 0, device = 0, nstreams = 1;
    // plugin parameters (XML keys of the reference)
    double alpha = 0.05;
    int limit = -1;
    int enable_thr = 1, thr = 15, enable_weight = 1, gray_variant = 0;
    // cv::BackgroundSubtractorMOG2 defaults (SURVEY 8a row a6)
    int history = 500;
    float Tb = 16.f, Tg = 9.f, TB = 0.9f, varInit = 15.f, varMin = 4.f, varMax = 75.f, CT = 0.05f, tau = 0.5f;
    int detect_shadows = 1, shadow_value = 127;
    bool host_bands_auto = true;   // "hostBands" not set: 3 bands when the background image goes back too, else 2 (1080p MOG2: 266 vs 274 us with the image, 176 vs 177 without; 4 bands 279 / 185)
    int host_bands = 2;        // row bands of the host-path upload/compute/download pipeline (1 = no overlap); 2 measured best at 1080p (277 vs 289 us with 4: each band costs ~8 host API calls)
    // AdaptiveSelectiveBackgroundLearning (defaults of its loadConfig, .cpp:121-125)
    int learning_frames = 90, asbl_counter = 0;
    int asbl_cur = 0;          // which of the two ASBL model buffers holds the model
    double alpha_learn = 0.05, alpha_detection = 0.05;
    // DPZivkovicAGMMBGS (defaults of its loadConfig, DPZivkovicAGMMBGS.cpp:97-100); its alpha default is set at create
    double dpz_threshold = 25.0;
    int gaussians = 3;
    // ... which the reference hands to the model ONCE, on the first frame (DPZivkovicAGMMBGS.cpp:58-65): later changes
    // of threshold / alpha / gaussians have no effect until the model is reset.  Latched copies used by the kernel:
    double dpz_thr_l = 25.0, dpz_alpha_l = 0.001;
    int dpz_K_l = 3;
    // DPAdaptiveMedianBGS / DPMeanBGS / DPWrenGABGS: "threshold" (kept in dpz_threshold), "alpha", "samplingRate",
    // "learningFrames"; handed to the model once, on the first frame, like DPZivkovic's (latched in dpz_thr_l / dpz_alpha_l)
    int sampling_rate = 7, sampling_rate_l = 7;
    // DPPratiMediodBGS: "historySize", "weight" (never used by the reference); latched copy, ring counters (the same for
    // every pixel because the wrapper clears the update mask), state block
    int history_size = 16, history_size_l = 16, prati_weight = 5;
    // SigmaDeltaBGS: "ampFactor", "minVar", "maxVar" (defaults of its loadConfig, SigmaDeltaBGS.cpp:68-70); applied before every frame
    int sd_amp = 1, sd_min_var = 15, sd_max_var = 255;
    int prati_n = 0, prati_pos = 0;
    uint8_t *d_prati = nullptr;
    size_t prati_bytes = 0;
    int abl_table = 1;         // ABL: 1 = lookup-table kernel, 0 = arithmetic kernel (A/B, identical results)
    int abl_blend = 0, lut_blend = 0;   // ABL: 0 = OpenCV 4.x fp64 addWeighted, 1 = OpenCV 2.4 fp32 addWeighted (table kernels only)
    int mog2_variant = 0;      // see launch_mog2 (mog2.cu): 0 production, 1 straight restatement, 8/9 timing instruments
    // geometry / counters
    int w = 0, h = 0, npx = 0;
    size_t pstride = 0;
    int64_t nframes = 0;
    int64_t mog2_epoch = 0;    // MOG2: the frame (counted in nframes) that last re-initialised the model (learningRate >= 1);
                               // the model's own frame counter, which drives the automatic learning rate, is nframes - mog2_epoch
    // device state
    float *d_state = nullptr;
    uint8_t *d_nmodes = nullptr;
    uint8_t *d_abl_lut = nullptr;         // ABL: 64 KB blend table for lut_alpha (simple_bgs.cu)
    double lut_alpha = -1.;
    uint8_t *d_hist[2] = {nullptr, nullptr};
    const uint8_t *hist_ptr[2] = {nullptr, nullptr};
    int have_hist = 0;
    // host-path staging
    uint8_t *d_ring[3] = {nullptr, nullptr, nullptr};
    int ring_pos = 0;
    uint8_t *d_fg = nullptr, *d_bg = nullptr;
    uint8_t *d_fan = nullptr;             // bgsb_process_fanout: the shared uploaded frame (owned by the first context)
    size_t d_fan_bytes = 0;
    cudaStream_t stream = nullptr;
    // host-path chunk pipeline: upload / compute / download overlap inside one synchronous call
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_up[8] = {}, ev_k[8] = {};
    // bgsb_submit / bgsb_wait: frames in flight, second output slot, download-complete events per slot
    uint8_t *d_fg2 = nullptr, *d_bg2 = nullptr;
    cudaEvent_t ev_dn[2] = {};
    uint64_t seq = 0;
    bool inflight = false;
    // the stream the model was last advanced on (see order_after_previous)
    cudaStream_t last_stream = nullptr;
    bool last_stream_set = false;
    cudaEvent_t ev_order = nullptr;
    int retain_input = 0;      // device path, FD / WMV / WMM: the caller's frames stay valid -> no history write-back
    // WMV quiet-group shortcut: wmv_bound[ew][r] = largest standard-deviation byte over all triples of range r for the
    // weight set ew (computed once per weight set on the device, launch_wmv_bound_table); wmv_quiet 0 switches it off
    int wmv_quiet = 1;
    int wmv_bound_valid[2] = {0, 0};
    unsigned char wmv_bound[2][256] = {};
    // per-call stage timing of the host path (FrameProcessor::tic / toc, FrameProcessor.cpp:484-494, per stage)
    int trace = 0;
    cudaEvent_t ev_t[6] = {};  // upload begin / end, kernels begin / end, download begin / end
    bgsb_trace last_trace = {};
};

static const char *algo_name(int algo)
{
    switch (algo) {
    case BGSB_ALGO_FRAME_DIFFERENCE: return "FrameDifferenceBGS";
    case BGSB_ALGO_STATIC_FRAME_DIFFERENCE: return "StaticFrameDifferenceBGS";
    case BGSB_ALGO_WEIGHTED_MOVING_MEAN: return "WeightedMovingMeanBGS";
    case BGSB_ALGO_WEIGHTED_MOVING_VARIANCE: return "WeightedMovingVarianceBGS";
    case BGSB_ALGO_MOG2: return "MixtureOfGaussianV2BGS";
    case BGSB_ALGO_ADAPTIVE_BG_LEARNING: return "AdaptiveBackgroundLearning";
    case BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING: return "AdaptiveSelectiveBackgroundLearning";
    case BGSB_ALGO_DP_ZIVKOVIC_AGMM: return "DPZivkovicAGMMBGS";
    case BGSB_ALGO_DP_ADAPTIVE_MEDIAN: return "DPAdaptiveMedianBGS";
    case BGSB_ALGO_DP_MEAN: return "DPMeanBGS";
    case BGSB_ALGO_DP_WREN_GA: return "DPWrenGABGS";
    case BGSB_ALGO_DP_PRATI_MEDIOD: return "DPPratiMediodBGS";
    case BGSB_ALGO_SIGMA_DELTA: return "SigmaDeltaBGS";
    }
    return "?";
}
static bool trace_env()
{
    static const bool on = [] { const char *e = getenv("BGSB_TRACE"); return e && e[0] && e[0] != '0'; }();
    return on;
}

static bool gmm_state(int algo);
static int dp_float_planes(int algo);
static void free_buffers(bgsb_ctx *c)
{
    cudaFree(c->d_state); c->d_state = nullptr;
    cudaFree(c->d_nmodes); c->d_nmodes = nullptr;
    cudaFree(c->d_abl_lut); c->d_abl_lut = nullptr; c->lut_alpha = -1.;
    for (int i = 0; i < 2; i++) { cudaFree(c->d_hist[i]); c->d_hist[i] = nullptr; c->hist_ptr[i] = nullptr; }
    for (int i = 0; i < 3; i++) { cudaFree(c->d_ring[i]); c->d_ring[i] = nullptr; }
    cudaFree(c->d_fg); c->d_fg = nullptr;
    cudaFree(c->d_bg); c->d_bg = nullptr;
    cudaFree(c->d_fg2); c->d_fg2 = nullptr;
    cudaFree(c->d_bg2); c->d_bg2 = nullptr;
    cudaFree(c->d_fan); c->d_fan = nullptr; c->d_fan_bytes = 0;
    cudaFree(c->d_prati); c->d_prati = nullptr; c->prati_bytes = 0; c->prati_n = c->prati_pos = 0;
    c->w = c->h = c->npx = 0; c->pstride = 0;
    c->nframes = 0; c->mog2_epoch = 0; c->have_hist = 0; c->ring_pos = 0;
}

// (Re)allocate model state for a geometry.  The reference discovers the frame size on the first
// process() call; cv::BackgroundSubtractorMOG2::operator() re-initialises when it changes.
static int ensure_geometry(bgsb_ctx *c, int w, int h)
{
    if (c->w == w && c->h == h) return BGSB_OK;
    BGSB_REQUIRE(w > 0 && h > 0, "empty frame");
    BGSB_REQUIRE((long long)w * h < (1LL << 30), "frame too large");
    BGSB_REQUIRE(!gmm_state(c->algo) || (long long)w * h <= (1LL << 27), "mixture-model frames are limited to 2^27 pixels");
    free_buffers(c);                              // geometry fields are 0 from here until every allocation has succeeded
    const int npx = w * h;
    const size_t pstride = ((size_t)npx + MOG2_TILE - 1) / MOG2_TILE * MOG2_TILE;       // whole state tiles
    const size_t S = (size_t)c->nstreams;
    cudaError_t e = cudaSuccess;
    if (gmm_state(c->algo)) {
        const size_t fb = S * MOG2_PLANES * pstride * sizeof(float);
        e = cudaMalloc(&c->d_state, fb);
        if (e == cudaSuccess) e = cudaMalloc(&c->d_nmodes, S * pstride);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_state, 0, fb, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_nmodes, 0, S * pstride, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    } else if (c->algo == BGSB_ALGO_DP_PRATI_MEDIOD) {
        // the state is sized by "historySize", which is handed over with the first frame: allocated there (launch_range)
    } else if (dp_float_planes(c->algo)) {
        e = cudaMalloc(&c->d_state, S * dp_float_planes(c->algo) * pstride * sizeof(float));      // written in full by the first frame
    } else {
        // ASBL: d_hist[0] = gray model, d_hist[1] = scratch (gray input + pre-median mask)
        // SigmaDelta: d_hist[0] = Mt, d_hist[1] = Vt
        int nh = (c->algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE || c->algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN ||
                  c->algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING || c->algo == BGSB_ALGO_SIGMA_DELTA) ? 2 : 1;
        for (int i = 0; i < nh && e == cudaSuccess; i++) e = cudaMalloc(&c->d_hist[i], S * npx * 3);
    }
    if (e != cudaSuccess) {                       // e.g. out of memory on a 2160p group: leave a context without geometry
        set_error("ensure_geometry(%d x %d x %d streams): %s", w, h, c->nstreams, cudaGetErrorString(e));
        (void)cudaGetLastError();
        free_buffers(c);
        return BGSB_ERR_CUDA;
    }
    c->w = w; c->h = h; c->npx = npx; c->pstride = pstride;
    return BGSB_OK;
}

// Staging buffers of the host paths; all-or-nothing like ensure_geometry.
static int staging_fail(bgsb_ctx *c, cudaError_t e)
{
    set_error("host staging (%d x %d x %d streams): %s", c->w, c->h, c->nstreams, cudaGetErrorString(e));
    (void)cudaGetLastError();
    for (int i = 0; i < 3; i++) { cudaFree(c->d_ring[i]); c->d_ring[i] = nullptr; }
    cudaFree(c->d_fg); c->d_fg = nullptr; cudaFree(c->d_bg); c->d_bg = nullptr;
    cudaFree(c->d_fg2); c->d_fg2 = nullptr; cudaFree(c->d_bg2); c->d_bg2 = nullptr;
    return BGSB_ERR_CUDA;
}

static int ensure_host_staging(bgsb_ctx *c)
{
    const size_t S = (size_t)c->nstreams;
    cudaError_t e = cudaSuccess;
    if (!c->d_ring[0]) {
        const bool two = (c->algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE || c->algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN);
        int nr = two ? 3 : (c->algo == BGSB_ALGO_FRAME_DIFFERENCE ? 2 : 1);
        for (int i = 0; i < nr && e == cudaSuccess; i++) e = cudaMalloc(&c->d_ring[i], S * c->npx * 3);
        c->ring_pos = 0;
    }
    if (e == cudaSuccess && !c->d_fg) e = cudaMalloc(&c->d_fg, S * c->npx);
    if (e == cudaSuccess && !c->d_bg && c->algo != BGSB_ALGO_FRAME_DIFFERENCE && c->algo != BGSB_ALGO_WEIGHTED_MOVING_VARIANCE)
        e = cudaMalloc(&c->d_bg, S * c->npx * 3);
    if (e != cudaSuccess) return staging_fail(c, e);
    return BGSB_OK;
}

// Host<->device image copy: a plain 1D copy when the host rows are dense (one DMA descriptor), a pitched
// copy otherwise (cv::Mat rows from cvQueryFrame are 4-byte aligned and may carry padding).
static cudaError_t copy_rows(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width, size_t rows,
                             cudaMemcpyKind kind, cudaStream_t st)
{
    if (dpitch == width && spitch == width) return cudaMemcpyAsync(dst, src, width * rows, kind, st);
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, kind, st);
}

static int warmup_frames(int algo)
{
    if (algo == BGSB_ALGO_FRAME_DIFFERENCE || algo == BGSB_ALGO_SIGMA_DELTA) return 1;
    if (algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE || algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN) return 2;
    return 0;
}
// a warm-up frame still needs a kernel: the model is initialised from it (FD / WMV / WMM just keep the uploaded frame)
static bool init_launch_on_warmup(int algo) { return algo == BGSB_ALGO_SIGMA_DELTA; }
// history images a plugin keeps: FD 1 (previous frame), WMV/WMM 2, ABL/StaticFD 1 (8-bit background)
static int history_images(int algo)
{
    if (algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE || algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN) return 2;
    return (gmm_state(algo) || dp_float_planes(algo) || algo == BGSB_ALGO_DP_PRATI_MEDIOD) ? 0 : 1;
}
// FD / WMV / WMM: the history is the previous input frame(s) -> on the host path it lives in the upload ring
static bool ring_history(int algo)
{
    return algo == BGSB_ALGO_FRAME_DIFFERENCE || algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE ||
           algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN;
}
// per-pixel mixture state in the MOG2 tile layout (d_state / d_nmodes)
static bool gmm_state(int algo) { return algo == BGSB_ALGO_MOG2 || algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM; }
// fp32 planes per pixel of the DP package's float models (d_state, [S][planes][pstride]): MeanBGS 3 means, WrenGA 3 means + variance
static int dp_float_planes(int algo) { return algo == BGSB_ALGO_DP_MEAN ? 3 : (algo == BGSB_ALGO_DP_WREN_GA ? 4 : 0); }
// channels of img_bgmodel: ASBL's model is the gray image (AdaptiveSelectiveBackgroundLearning.cpp:103)
static int bg_channels(int algo) { return algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING ? 1 : 3; }
// the mask depends on neighbouring pixels (3x3 median): no row-band sub-launches
// (DPPratiMediod: its mask is the hysteresis of two thresholds over the 8 neighbours)
static bool stencil_algo(int algo) { return algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING || algo == BGSB_ALGO_DP_PRATI_MEDIOD; }
static bool writes_background(int algo)
{
    return algo == BGSB_ALGO_MOG2 || algo == BGSB_ALGO_ADAPTIVE_BG_LEARNING || algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING ||
           algo == BGSB_ALGO_STATIC_FRAME_DIFFERENCE || algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN;
}

// Advance the model by T frames that sit in device memory.  `own_history`: write FD/WMV history
// into the context's own buffers (caller's frame buffers may be reused after the call).
// Launch the kernel for pixels [p0, p0+pcount) of the frame(s); p0 must be a multiple of 64 (a MOG2 state tile).
// A sub-range is only used for single-stream, single-frame calls (host-path chunk pipelining).
static int launch_range(bgsb_ctx *c, const uint8_t *d_frames, int T, uint8_t *d_fg, uint8_t *d_bg,
                        int bg_last_only, bool own_history, cudaStream_t stream, size_t p0, int pcount,
                        unsigned *d_bits = nullptr, int bit_thr = 0)
{
    if (c->algo == BGSB_ALGO_MOG2) {
        BGSB_REQUIRE(T <= MOG2_TMAX, "temporal batch too long (max 32)");
        // learningRate >= 1: cv::BackgroundSubtractorMOG2::apply re-initialises the model before every such frame
        // (needToInitialize), so each frame starts from an empty model with nframes = 1.  No frame can reuse another's
        // state: a batch runs one frame per launch, and a group one stream per launch too (a launch's streams sit L.T
        // frames apart in the batch layouts).
        const bool reinit = c->alpha >= 1;
        // Short batches of one stream run frame by frame: the T == 1 kernel costs less per frame than the
        // temporal-fusion kernel's fixed state load/store until about six frames share it (profiles/).
        const bool per_frame = T > 1 && ((T < 6 && c->nstreams == 1 && c->mog2_variant == 0) || reinit);
        const bool per_stream = per_frame && c->nstreams > 1;
        const int nlaunch = per_frame ? T : 1, Tl = per_frame ? 1 : T;
        const int nsplit = per_stream ? c->nstreams : 1, Sl = per_stream ? 1 : c->nstreams;
        // frames the model has seen since it was last (re)initialised (OpenCV's nframes)
        const int64_t seen = c->nframes - c->mog2_epoch;
        // MOG2Invoker: varMin = min(_varMin, _varMax), varMax = max(_varMin, _varMax)
        const float vmin = std::min(c->varMin, c->varMax), vmax = std::max(c->varMin, c->varMax);
        for (int s = 0; s < nsplit; s++)
        for (int i = 0; i < nlaunch; i++) {
            Mog2Launch L;
            memset(&L, 0, sizeof(L));
            const size_t f0 = ((size_t)s * T + i) * c->npx;        // first pixel of frame i of stream s in the batch buffers
            L.frames = d_frames + (f0 + p0) * 3; L.fg = d_fg ? d_fg + f0 + p0 : nullptr;
            L.bg = nullptr;
            if (d_bits) {                                  // whole single frames on the production kernel only (ctx_process_frame)
                L.bits = d_bits; L.w = c->w; L.wpr = (c->w + 31) / 32; L.bits_stride = (size_t)L.wpr * c->h; L.bit_thr = bit_thr;
            }
            if (d_bg) {
                if (!per_frame) L.bg = d_bg + p0 * 3;
                else if (!bg_last_only) L.bg = d_bg + (f0 + p0) * 3;
                else if (i == T - 1) L.bg = d_bg + ((size_t)s * c->npx + p0) * 3;
            }
            L.state = c->d_state + ((size_t)s * c->pstride + p0) * MOG2_PLANES;   // p0 % 64 == 0
            L.nmodes = c->d_nmodes + (size_t)s * c->pstride + p0; L.pstride = c->pstride;
            L.npx = pcount; L.T = Tl; L.bg_last_only = per_frame ? 0 : bg_last_only;
            L.fresh = reinit || seen + i == 0;
            L.fast_ok = 1;
            L.one = 1.f;
            L.enable_thr = c->enable_thr; L.thr = c->thr;
            L.detect_shadows = c->detect_shadows; L.shadow_value = c->shadow_value;
            L.Tb = c->Tb; L.Tg = c->Tg; L.TB = c->TB; L.varInit = c->varInit; L.varMin = vmin;
            L.varMax = vmax; L.tau = c->tau;
            for (int t = 0; t < Tl; t++) {
                // operator(): ++nframes; learningRate = alpha>=0 && nframes>1 ? alpha : 1./min(2*nframes, history)
                int64_t nf = reinit ? 1 : seen + i + t + 1;
                double lr = (c->alpha >= 0 && nf > 1) ? c->alpha : 1. / (double)std::min<int64_t>(2 * nf, c->history);
                L.alphaT[t] = (float)lr;
                L.alpha1[t] = 1.f - L.alphaT[t];
                L.prune[t] = (float)(-lr * (double)c->CT);
                if (!(L.alphaT[t] >= 1e-4f && L.alphaT[t] <= 1.f)) L.fast_ok = 0;
            }
            int rc = launch_mog2(L, Sl, c->mog2_variant, stream);
            if (rc) return rc;
        }
        if (reinit) c->mog2_epoch = c->nframes + T - 1;  // the last frame of the batch re-initialised the model
    } else if (c->algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM) {
        for (int t = 0; t < T; t++) {
            DpzLaunch L;
            memset(&L, 0, sizeof(L));
            // batch layouts: frames [S][T][npx*3], masks [S][T][npx]; pixels [p0, p0+pcount), p0 on a state tile
            L.frame = d_frames + ((size_t)t * c->npx + p0) * 3; L.frame_stride = (size_t)T * c->npx * 3;
            L.fg = d_fg + (size_t)t * c->npx + p0; L.fg_stride = (size_t)T * c->npx;
            L.state = c->d_state + p0 * MOG2_PLANES; L.nmodes = c->d_nmodes + p0; L.pstride = c->pstride;
            if (c->nframes + t == 0 && p0 == 0) { c->dpz_thr_l = c->dpz_threshold; c->dpz_alpha_l = c->alpha; c->dpz_K_l = c->gaussians; }
            L.npx = pcount; L.K = c->dpz_K_l;
            L.fresh = (c->nframes + t == 0);
            L.low_thr = (float)c->dpz_thr_l; L.alpha = (float)c->dpz_alpha_l;
            int rc = launch_dpz(L, c->nstreams, stream);
            if (rc) return rc;
        }
    } else if (c->algo == BGSB_ALGO_DP_ADAPTIVE_MEDIAN || c->algo == BGSB_ALGO_DP_MEAN || c->algo == BGSB_ALGO_DP_WREN_GA) {
        for (int t = 0; t < T; t++) {
            DpsLaunch L;
            memset(&L, 0, sizeof(L));
            const int64_t frame_num = c->nframes + t;                      // the wrappers' frameNumber
            if (frame_num == 0 && p0 == 0) { c->dpz_thr_l = c->dpz_threshold; c->dpz_alpha_l = c->alpha; c->sampling_rate_l = c->sampling_rate; }
            L.kind = c->algo == BGSB_ALGO_DP_ADAPTIVE_MEDIAN ? DPS_MEDIAN : (c->algo == BGSB_ALGO_DP_MEAN ? DPS_MEAN : DPS_WREN);
            L.frame = d_frames + ((size_t)t * c->npx + p0) * 3; L.frame_stride = (size_t)T * c->npx * 3;
            L.fg = d_fg + (size_t)t * c->npx + p0; L.fg_stride = (size_t)T * c->npx;
            L.pstride = c->pstride;
            if (L.kind == DPS_MEDIAN) { L.median = c->d_hist[0] + p0 * 3; L.median_stride = (size_t)c->npx * 3; }
            else L.state = c->d_state + p0;
            L.npx = pcount; L.fresh = frame_num == 0;
            if (L.kind == DPS_MEDIAN) {
                // thresholds are unsigned char members: high = (uchar)(2 * (uchar)threshold) (AdaptiveMedianBGS.h:49-50)
                const unsigned char low = (unsigned char)(int)c->dpz_thr_l;
                L.high_u = (unsigned char)(2 * low);
                L.update = (frame_num % c->sampling_rate_l) == 1;          // AdaptiveMedianBGS.cpp:67
            } else if (L.kind == DPS_MEAN) {
                const unsigned low = (unsigned)(int)c->dpz_thr_l;          // unsigned int members (MeanBGS.h:47-48)
                L.high_f = (float)(2u * low);
            } else {
                const float low = (float)c->dpz_thr_l;                     // float members (WrenGA.h:48-49)
                L.high_f = 2 * low;
            }
            L.alpha = (float)c->dpz_alpha_l; L.one_minus_alpha = 1.0f - L.alpha;
            int rc = launch_dp_simple(L, c->nstreams, stream);
            if (rc) return rc;
        }
    } else if (c->algo == BGSB_ALGO_SIGMA_DELTA) {
        for (int t = 0; t < T; t++) {
            SdLaunch L;
            memset(&L, 0, sizeof(L));
            const int64_t frame_num = c->nframes + t;
            L.frame = d_frames + ((size_t)t * c->npx + p0) * 3; L.frame_stride = (size_t)T * c->npx * 3;
            L.first = frame_num == 0;                                      // SigmaDeltaBGS.cpp:28-33: initialise, no output
            L.fg = (d_fg && !L.first) ? d_fg + (size_t)t * c->npx + p0 : nullptr; L.fg_stride = (size_t)T * c->npx;
            L.Mt = c->d_hist[0] + p0 * 3; L.Vt = c->d_hist[1] + p0 * 3; L.model_stride = (size_t)c->npx * 3;
            L.npx = pcount; L.w = c->w; L.p0 = (long long)p0;
            // uint32_t parameters; the clamp goes through uint8_t helpers (sdLaMa091.cpp:62-63, :581)
            L.N = (unsigned)c->sd_amp; L.vmin8 = (unsigned)c->sd_min_var & 0xffu; L.vmax8 = (unsigned)c->sd_max_var & 0xffu;
            int rc = launch_sigma_delta(L, c->nstreams, stream);
            if (rc) return rc;
        }
    } else if (c->algo == BGSB_ALGO_DP_PRATI_MEDIOD) {
        BGSB_REQUIRE(p0 == 0 && pcount == c->npx, "DPPratiMediod works on whole frames (8-neighbour hysteresis)");
        for (int t = 0; t < T; t++) {
            const int64_t frame_num = c->nframes + t;                      // the wrapper's frameNumber
            if (frame_num == 0) {                                          // DPPratiMediodBGS.cpp:57-62, once
                c->dpz_thr_l = c->dpz_threshold; c->sampling_rate_l = c->sampling_rate; c->history_size_l = c->history_size;
                c->prati_n = 0; c->prati_pos = 0;
            }
            PratiLaunch L;
            memset(&L, 0, sizeof(L));
            prati_layout(c->npx, c->history_size_l, &L.plane3, &L.plane1, &L.stream_bytes);
            const size_t need = L.stream_bytes * (size_t)c->nstreams;
            if (!c->d_prati || c->prati_bytes < need) {
                BGSB_REQUIRE(frame_num == 0, "DPPratiMediod: state missing");
                cudaFree(c->d_prati); c->d_prati = nullptr; c->prati_bytes = 0;
                BGSB_CUDA(cudaMalloc(&c->d_prati, need));
                c->prati_bytes = need;
            }
            L.frame = d_frames + (size_t)t * c->npx * 3; L.frame_stride = (size_t)T * c->npx * 3;
            L.fg = d_fg + (size_t)t * c->npx; L.fg_stride = (size_t)T * c->npx;
            L.state = c->d_prati;
            L.w = c->w; L.h = c->h; L.H = c->history_size_l; L.n = c->prati_n; L.pos = c->prati_pos;
            L.low = (unsigned)(int)c->dpz_thr_l; L.high = 2u * L.low;      // unsigned int members (PratiMediodBGS.h:52-53)
            if (frame_num < c->history_size_l) {                           // Subtract :239-244: both masks cleared
                for (int s = 0; s < c->nstreams; s++)
                    BGSB_CUDA(cudaMemsetAsync(L.fg + (size_t)s * L.fg_stride, 0, (size_t)c->npx, stream));
            } else {
                int rc = launch_prati_subtract(L, c->nstreams, stream);
                if (rc) return rc;
            }
            if (frame_num % c->sampling_rate_l == 0) {                     // Update :73
                int rc = launch_prati_update(L, c->nstreams, stream);
                if (rc) return rc;
                if (c->prati_n == c->history_size_l) c->prati_pos = (c->prati_pos + 1) % c->history_size_l;
                else { c->prati_n++; c->prati_pos = 0; }
            }
        }
    } else if (c->algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING) {
        BGSB_REQUIRE(p0 == 0 && pcount == c->npx, "ASBL works on whole frames (3x3 median)");
        const size_t npx = (size_t)c->npx;
        for (int t = 0; t < T; t++) {
            AsblLaunch L;
            memset(&L, 0, sizeof(L));
            // batch layouts: frames [S][T][npx*3], masks [S][T][npx], model images [S][T][npx] or [S][npx]
            L.frame = d_frames + (size_t)t * npx * 3; L.frame_stride = (size_t)T * npx * 3;
            L.fg = d_fg + (size_t)t * npx; L.fg_stride = (size_t)T * npx;
            if (d_bg && (!bg_last_only || t == T - 1)) {
                L.bgout = bg_last_only ? d_bg : d_bg + (size_t)t * npx;
                L.bg_stride = bg_last_only ? npx : (size_t)T * npx;
            }
            // d_hist[1] (3 bytes per pixel) = gray scratch | pre-median mask scratch | second model buffer
            uint8_t *const mbuf[2] = {c->d_hist[0], c->d_hist[1] + 2 * (size_t)c->nstreams * npx};
            L.model = mbuf[c->asbl_cur]; L.model_out = mbuf[c->asbl_cur ^ 1];
            L.gray = c->d_hist[1]; L.raw = c->d_hist[1] + (size_t)c->nstreams * npx;
            L.w = c->w; L.h = c->h;
            L.first = (c->have_hist == 0 && t == 0);
            // learning phase: `learningFrames > 0 && counter <= learningFrames`, counter++ (.cpp:65-71)
            const bool learning = c->learning_frames > 0 && c->asbl_counter <= c->learning_frames;
            if (learning) c->asbl_counter++;
            L.selective = learning ? 0 : 1;
            L.alpha = learning ? c->alpha_learn : c->alpha_detection;
            L.thr = c->thr; L.gray_variant = c->gray_variant;
            // the blend of two bytes as a 64 KB table (ABL's, simple_bgs.cu): rebuilt when alpha changes, i.e. once at
            // the end of the learning phase; stream-ordered before the kernel that reads it
            if (!c->d_abl_lut) BGSB_CUDA(cudaMalloc(&c->d_abl_lut, ABL_LUT_BYTES));
            if (c->lut_alpha != L.alpha) {
                int rcl = launch_abl_lut_build(c->d_abl_lut, L.alpha, 0, stream);
                if (rcl) return rcl;
                c->lut_alpha = L.alpha;
            }
            L.lut = c->d_abl_lut;
            int swapped = 0;
            int rc = launch_asbl(L, c->nstreams, stream, &swapped);
            if (rc) return rc;
            c->asbl_cur ^= swapped;
            if (t == 0 && c->have_hist == 0) c->have_hist = 1;   // the model exists from the first frame on
        }
    } else {
        SimpleLaunch L;
        memset(&L, 0, sizeof(L));
        L.one = 1.f;
        L.frames = d_frames + p0 * 3; L.fg = d_fg + p0; L.bg = d_bg ? d_bg + p0 * 3 : nullptr;
        L.hist0 = c->hist_ptr[0] ? c->hist_ptr[0] + p0 * 3 : nullptr;
        L.hist1 = c->hist_ptr[1] ? c->hist_ptr[1] + p0 * 3 : nullptr;
        L.hist0_out = (own_history && c->d_hist[0]) ? c->d_hist[0] + p0 * 3 : nullptr;
        L.hist1_out = (own_history && c->d_hist[1]) ? c->d_hist[1] + p0 * 3 : nullptr;
        if (c->algo == BGSB_ALGO_ADAPTIVE_BG_LEARNING || c->algo == BGSB_ALGO_STATIC_FRAME_DIFFERENCE) {
            L.hist0 = c->d_hist[0] + p0 * 3; L.hist0_out = c->d_hist[0] + p0 * 3;    // the 8-bit background model
        }
        L.npx = pcount; L.T = T; L.have_hist = c->have_hist; L.bg_last_only = bg_last_only;
        L.enable_thr = c->enable_thr; L.thr = c->thr; L.gray_variant = c->gray_variant;
        L.alpha = c->alpha;
        if (c->algo == BGSB_ALGO_ADAPTIVE_BG_LEARNING && c->abl_table) {
            if (!c->d_abl_lut) BGSB_CUDA(cudaMalloc(&c->d_abl_lut, ABL_LUT_BYTES));
            if (c->lut_alpha != c->alpha || c->lut_blend != c->abl_blend) {     // stream-ordered before the kernel that reads it
                int rcl = launch_abl_lut_build(c->d_abl_lut, c->alpha, c->abl_blend, stream);
                if (rcl) return rcl;
                c->lut_alpha = c->alpha; c->lut_blend = c->abl_blend;
            }
            L.abl_lut = c->d_abl_lut;
            L.abl_lut_mode = c->abl_table == 2 ? 1 : (c->abl_table == 3 ? 2 : 0);
            L.abl_quiet = c->wmv_quiet;
        }
        L.abl_update = (c->limit == -1);   // the limit>0 branch never fires: counter stays 0 (.cpp:52,60-61)
        if (c->enable_weight) { L.w0 = 0.5; L.w1 = 0.3; L.w2 = 0.2; }      // WeightedMovingVarianceBGS.cpp:67-68
        else { L.w0 = 0.3; L.w1 = 0.3; L.w2 = 0.3; }                          // :70
        L.quiet_range = -1;
        if (c->algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE && c->wmv_quiet && c->enable_thr && c->thr >= 0) {
            const int ew = c->enable_weight ? 1 : 0;
            if (!c->wmv_bound_valid[ew]) {          // once per weight set: 2^24 triples through the kernel's own routine
                unsigned *d_tab = nullptr, h_tab[256];
                BGSB_CUDA(cudaMalloc(&d_tab, sizeof(h_tab)));
                int rct = launch_wmv_bound_table(d_tab, L.w0, L.w1, L.w2, stream);
                cudaError_t e = rct ? cudaErrorUnknown : cudaMemcpyAsync(h_tab, d_tab, sizeof(h_tab), cudaMemcpyDeviceToHost, stream);
                if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
                cudaFree(d_tab);
                if (rct) return rct;
                BGSB_CUDA(e);
                for (int r = 0; r < 256; r++) c->wmv_bound[ew][r] = (unsigned char)std::min(255u, h_tab[r]);
                c->wmv_bound_valid[ew] = 1;
            }
            // the largest range R such that every triple of range <= R stays at or below the threshold
            int R = -1;
            while (R + 1 < 256 && (int)c->wmv_bound[ew][R + 1] <= c->thr) R++;
            L.quiet_range = R;
        }
        int rc = launch_simple(c->algo, L, c->nstreams, stream);
        if (rc) return rc;
    }
    return BGSB_OK;
}

// The model (d_state, d_hist, the blend table) is advanced by kernels on ONE stream per call: the caller's for the
// *_dev entry points, the context's own for the host-buffer ones.  When a call arrives on a different stream than the
// previous one, it is ordered behind it (an event recorded now on the previous stream covers everything that call
// enqueued there).  A stream handed to a *_dev call must therefore stay alive until the next call on this context;
// if it was destroyed the library falls back to a device synchronisation.
static int order_after_previous(bgsb_ctx *c, cudaStream_t next)
{
    if (c->last_stream_set && c->last_stream != next) {
        if (!c->ev_order) BGSB_CUDA(cudaEventCreateWithFlags(&c->ev_order, cudaEventDisableTiming));
        cudaError_t e = cudaEventRecord(c->ev_order, c->last_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(next, c->ev_order, 0);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            BGSB_CUDA(cudaDeviceSynchronize());
        }
    }
    c->last_stream = next; c->last_stream_set = true;
    return BGSB_OK;
}

// Bookkeeping after T frames went through launch_range.
static void advance(bgsb_ctx *c, int T, bool own_history)
{
    if (c->algo != BGSB_ALGO_MOG2 && own_history) {
        int need = history_images(c->algo);
        c->have_hist = (int)std::min<int64_t>(need, (int64_t)c->have_hist + T);
        c->hist_ptr[0] = c->d_hist[0]; c->hist_ptr[1] = c->d_hist[1];
    }
    c->nframes += T;
}

// Advance the model by T frames that sit in device memory.  `own_history`: write FD/WMV history
// into the context's own buffers (caller's frame buffers may be reused after the call).
static int run_frames(bgsb_ctx *c, const uint8_t *d_frames, int T, uint8_t *d_fg, uint8_t *d_bg,
                      int bg_last_only, bool own_history, cudaStream_t stream)
{
    int rc = launch_range(c, d_frames, T, d_fg, d_bg, bg_last_only, own_history, stream, 0, c->npx);
    if (rc) return rc;
    advance(c, T, own_history);
    return BGSB_OK;
}

namespace bgsb {
int sm_count(int device)
{
    static std::atomic<int> cached[64];
    if (device < 0 || device >= 64) return 148;
    int v = cached[device].load(std::memory_order_relaxed);
    if (v <= 0) {
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
        cached[device].store(v, std::memory_order_relaxed);
    }
    return v;
}

bool pdl_enabled()
{
    static const bool on = [] { const char *e = getenv("BGSB_NO_PDL"); return !(e && e[0] == '1'); }();
    return on;
}
}  // namespace bgsb

// copy streams and per-band events of the upload / kernel / download pipelines
static int ensure_pipe_streams(bgsb_ctx *c)
{
    if (c->s_h2d) return BGSB_OK;
    BGSB_CUDA(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    BGSB_CUDA(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) {
        BGSB_CUDA(cudaEventCreateWithFlags(&c->ev_up[i], cudaEventDisableTiming));
        BGSB_CUDA(cudaEventCreateWithFlags(&c->ev_k[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 2; i++) BGSB_CUDA(cudaEventCreateWithFlags(&c->ev_dn[i], cudaEventDisableTiming));
    return BGSB_OK;
}

// Frames queued by bgsb_submit: every other entry point that touches the model or the staging buffers first waits
// for them (results are then in the host buffers given to bgsb_submit).
static int drain(bgsb_ctx *c)
{
    if (!c->inflight) return BGSB_OK;
    BGSB_CUDA(cudaSetDevice(c->device));
    BGSB_CUDA(cudaStreamSynchronize(c->s_h2d));
    BGSB_CUDA(cudaStreamSynchronize(c->stream));
    BGSB_CUDA(cudaStreamSynchronize(c->s_d2h));
    c->inflight = false;
    return BGSB_OK;
}

extern "C" {

const char *bgsb_last_error(void) { return bgsb::g_err; }
const char *bgsb_version(void) { return "bgsb200 0.1 (sm_100a)"; }
uint64_t bgsb_kernel_launch_count(void) { return bgsb::g_launches.load(); }

int bgsb_host_alloc(void **ptr, size_t bytes, int write_combined)
{
    BGSB_REQUIRE(ptr && bytes > 0, "bad args");
    BGSB_CUDA(cudaHostAlloc(ptr, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
    return BGSB_OK;
}

void bgsb_host_free(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
}

int bgsb_device_count(int *count)
{
    BGSB_REQUIRE(count, "null");
    BGSB_CUDA(cudaGetDeviceCount(count));
    return BGSB_OK;
}

int bgsb_create_group(bgsb_ctx **out, int algo, int device, int nstreams)
{
    BGSB_REQUIRE(out, "null out");
    BGSB_REQUIRE(algo == BGSB_ALGO_FRAME_DIFFERENCE || algo == BGSB_ALGO_WEIGHTED_MOVING_VARIANCE ||
                 algo == BGSB_ALGO_MOG2 || algo == BGSB_ALGO_ADAPTIVE_BG_LEARNING ||
                 algo == BGSB_ALGO_STATIC_FRAME_DIFFERENCE || algo == BGSB_ALGO_WEIGHTED_MOVING_MEAN || algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING ||
                 algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM || algo == BGSB_ALGO_DP_ADAPTIVE_MEDIAN || algo == BGSB_ALGO_DP_MEAN ||
                 algo == BGSB_ALGO_DP_WREN_GA || algo == BGSB_ALGO_DP_PRATI_MEDIOD || algo == BGSB_ALGO_SIGMA_DELTA,
                 "unknown algorithm id (USTC_BGS ids: 0 FD, 1 StaticFD, 2 WMM, 3 WMV, 5 MOG2, 6 ABL, 7 ASBL, 9 DPAdaptiveMedian, "
                 "11 DPZivkovicAGMM, 12 DPMean, 13 DPWrenGA, 14 DPPratiMediod, 35 SigmaDelta)");
    BGSB_REQUIRE(nstreams >= 1 && nstreams <= 65535, "nstreams out of range");
    BGSB_CUDA(cudaSetDevice(device));
    bgsb_ctx *c = new bgsb_ctx();
    c->algo = algo; c->device = device; c->nstreams = nstreams;
    if (algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING) c->thr = 25;        // loadConfig default (.cpp:124)
    if (algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM) c->alpha = 0.001;                        // DPZivkovicAGMMBGS.cpp:98
    // loadConfig defaults of the DP wrappers (DPAdaptiveMedianBGS.cpp:101-103, DPMeanBGS.cpp:103-105, DPWrenGABGS.cpp:103-105);
    // the real-valued ones are float literals read into doubles
    if (algo == BGSB_ALGO_DP_ADAPTIVE_MEDIAN) { c->dpz_threshold = 40; c->thr = 40; c->sampling_rate = 7; c->learning_frames = 30; }
    if (algo == BGSB_ALGO_DP_MEAN) { c->dpz_threshold = 2700; c->thr = 2700; c->alpha = (double)1e-6f; c->learning_frames = 30; }
    if (algo == BGSB_ALGO_DP_PRATI_MEDIOD) { c->dpz_threshold = 30; c->thr = 30; c->sampling_rate = 5; }   // DPPratiMediodBGS.cpp:104-107
    if (algo == BGSB_ALGO_DP_WREN_GA) { c->dpz_threshold = (double)12.25f; c->thr = 12; c->alpha = (double)0.005f; c->learning_frames = 30; }
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate -> %s", cudaGetErrorString(e));
        delete c;
        return BGSB_ERR_CUDA;
    }
    *out = c;
    return BGSB_OK;
}

int bgsb_create(bgsb_ctx **out, int algo, int device) { return bgsb_create_group(out, algo, device, 1); }

void bgsb_destroy(bgsb_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    drain(c);
    if (c->stream) { cudaStreamSynchronize(c->stream); }
    free_buffers(c);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    for (int i = 0; i < 8; i++) { if (c->ev_up[i]) cudaEventDestroy(c->ev_up[i]); if (c->ev_k[i]) cudaEventDestroy(c->ev_k[i]); }
    for (int i = 0; i < 2; i++) if (c->ev_dn[i]) cudaEventDestroy(c->ev_dn[i]);
    if (c->ev_order) cudaEventDestroy(c->ev_order);
    for (int i = 0; i < 6; i++) if (c->ev_t[i]) cudaEventDestroy(c->ev_t[i]);
    delete c;
}

int bgsb_reset(bgsb_ctx *c)
{
    BGSB_REQUIRE(c, "null ctx");
    int rc = drain(c);
    if (rc) return rc;
    c->nframes = 0; c->mog2_epoch = 0; c->have_hist = 0; c->asbl_counter = 0;
    c->hist_ptr[0] = c->hist_ptr[1] = nullptr;
    return BGSB_OK;
}

int bgsb_set_param(bgsb_ctx *c, const char *key, double v)
{
    BGSB_REQUIRE(c && key, "null");
    std::string k(key);
    if (k == "alpha") c->alpha = v;
    else if (k == "limit") c->limit = (int)v;
    else if (k == "learningFrames") c->learning_frames = (int)v;
    else if (k == "samplingRate") { BGSB_REQUIRE(v >= 1 && v <= (double)(1 << 30), "samplingRate must be positive"); c->sampling_rate = (int)v; }
    else if (k == "historySize") { BGSB_REQUIRE(v >= 1 && v <= 64, "historySize in [1,64]"); c->history_size = (int)v; }
    else if (k == "ampFactor") { BGSB_REQUIRE(v >= 0 && v <= 16777216., "ampFactor out of range"); c->sd_amp = (int)v; }
    else if (k == "minVar") { BGSB_REQUIRE(v >= 0 && v <= 2147483647., "minVar out of range"); c->sd_min_var = (int)v; }
    else if (k == "maxVar") { BGSB_REQUIRE(v >= 0 && v <= 2147483647., "maxVar out of range"); c->sd_max_var = (int)v; }
    else if (k == "weight") c->prati_weight = (int)v;                        // stored for the XML round trip; the reference never reads it
    else if (k == "alphaLearn") c->alpha_learn = v;
    else if (k == "alphaDetection") c->alpha_detection = v;
    else if (k == "enableThreshold") c->enable_thr = (v != 0);
    else if (k == "threshold") { c->thr = (int)v; c->dpz_threshold = v; }      // DPZivkovicAGMM keeps the real value
    else if (k == "gaussians") { BGSB_REQUIRE(v >= 1 && v <= MOG2_K, "gaussians in [1,5]"); c->gaussians = (int)v; }
    else if (k == "enableWeight") c->enable_weight = (v != 0);
    else if (k == "grayVariant") { BGSB_REQUIRE(v == 0 || v == 1, "grayVariant is 0 or 1"); c->gray_variant = (int)v; }
    else if (k == "history") { BGSB_REQUIRE(v >= 1, "history >= 1"); c->history = (int)v; }
    else if (k == "nmixtures") { BGSB_REQUIRE((int)v == MOG2_K, "nmixtures is fixed at 5"); }
    else if (k == "varThreshold") c->Tb = (float)v;
    else if (k == "varThresholdGen") c->Tg = (float)v;
    else if (k == "backgroundRatio") c->TB = (float)v;
    else if (k == "varInit") c->varInit = (float)v;
    else if (k == "varMin") c->varMin = (float)v;
    else if (k == "varMax") c->varMax = (float)v;
    else if (k == "complexityReductionThreshold") c->CT = (float)v;
    else if (k == "detectShadows") c->detect_shadows = (v != 0);
    else if (k == "shadowValue") c->shadow_value = (int)v;
    else if (k == "shadowThreshold") c->tau = (float)v;
    else if (k == "hostBands") { BGSB_REQUIRE(v >= 1 && v <= 8, "hostBands in [1,8]"); c->host_bands = (int)v; c->host_bands_auto = false; }
    else if (k == "retainInput") c->retain_input = (v != 0);
    else if (k == "quietGroups") c->wmv_quiet = (v != 0);
    else if (k == "trace") c->trace = (v != 0);
#ifdef BGSB_INSTRUMENT
    else if (k == "kernelVariant") { BGSB_REQUIRE(v == 0 || v == 1 || v == 8 || v == 9, "kernelVariant is 0 or 1 (8, 9: timing instruments)"); c->mog2_variant = (int)v; }
#else
    else if (k == "kernelVariant") { BGSB_REQUIRE(v == 0 || v == 1, "kernelVariant is 0 or 1"); c->mog2_variant = (int)v; }
#endif
    else if (k == "ablTable") {
        BGSB_REQUIRE(v == 0 || v == 1 || v == 2 || v == 3, "ablTable is 0, 1, 2 or 3");
        BGSB_REQUIRE(v != 0 || c->abl_blend == 0, "the OpenCV 2.4 blend (ablBlend 1) exists in table form only");
        c->abl_table = (int)v;
    }
    else if (k == "ablBlend") {
        BGSB_REQUIRE(v == 0 || v == 1, "ablBlend is 0 (OpenCV 4.x, fp64) or 1 (OpenCV 2.4, fp32)");
        BGSB_REQUIRE(v == 0 || c->abl_table != 0, "the OpenCV 2.4 blend (ablBlend 1) exists in table form only");
        c->abl_blend = (int)v;
    }
    else if (k == "showOutput" || k == "showForeground" || k == "showBackground") { /* GUI only */ }
    else { set_error("bgsb_set_param: unknown key '%s'", key); return BGSB_ERR_ARG; }
    return BGSB_OK;
}

int bgsb_get_param(bgsb_ctx *c, const char *key, double *v)
{
    BGSB_REQUIRE(c && key && v, "null");
    std::string k(key);
    if (k == "alpha") *v = c->alpha;
    else if (k == "limit") *v = c->limit;
    else if (k == "learningFrames") *v = c->learning_frames;
    else if (k == "alphaLearn") *v = c->alpha_learn;
    else if (k == "alphaDetection") *v = c->alpha_detection;
    else if (k == "enableThreshold") *v = c->enable_thr;
    else if (k == "threshold") *v = (c->algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM || c->algo == BGSB_ALGO_DP_WREN_GA) ? c->dpz_threshold : c->thr;
    else if (k == "samplingRate") *v = c->sampling_rate;
    else if (k == "historySize") *v = c->history_size;
    else if (k == "ampFactor") *v = c->sd_amp;
    else if (k == "minVar") *v = c->sd_min_var;
    else if (k == "maxVar") *v = c->sd_max_var;
    else if (k == "weight") *v = c->prati_weight;
    else if (k == "gaussians") *v = c->gaussians;
    else if (k == "enableWeight") *v = c->enable_weight;
    else if (k == "grayVariant") *v = c->gray_variant;
    else if (k == "history") *v = c->history;
    else if (k == "nmixtures") *v = MOG2_K;
    else if (k == "varThreshold") *v = c->Tb;
    else if (k == "varThresholdGen") *v = c->Tg;
    else if (k == "backgroundRatio") *v = c->TB;
    else if (k == "varInit") *v = c->varInit;
    else if (k == "varMin") *v = c->varMin;
    else if (k == "varMax") *v = c->varMax;
    else if (k == "complexityReductionThreshold") *v = c->CT;
    else if (k == "detectShadows") *v = c->detect_shadows;
    else if (k == "shadowValue") *v = c->shadow_value;
    else if (k == "shadowThreshold") *v = c->tau;
    else if (k == "kernelVariant") *v = c->mog2_variant;
    else if (k == "hostBands") *v = c->host_bands;
    else if (k == "retainInput") *v = c->retain_input;
    else if (k == "quietGroups") *v = c->wmv_quiet;
    else if (k == "trace") *v = c->trace;
    else if (k == "ablTable") *v = c->abl_table;
    else if (k == "ablBlend") *v = c->abl_blend;
    else { set_error("bgsb_get_param: unknown key '%s'", key); return BGSB_ERR_ARG; }
    return BGSB_OK;
}

int bgsb_trace_last(bgsb_ctx *c, bgsb_trace *out)
{
    BGSB_REQUIRE(c && out, "null");
    if (!c->ev_t[0]) { set_error("bgsb_trace_last: no traced bgsb_process call yet (set the \"trace\" parameter or BGSB_TRACE=1)"); return BGSB_ERR_STATE; }
    *out = c->last_trace;
    return BGSB_OK;
}

int bgsb_frame_count(bgsb_ctx *c, int64_t *n)
{
    BGSB_REQUIRE(c && n, "null");
    *n = c->nframes;
    return BGSB_OK;
}

int bgsb_state_bytes(bgsb_ctx *c, size_t *bytes)
{
    BGSB_REQUIRE(c && bytes, "null");
    if (c->algo == BGSB_ALGO_MOG2) *bytes = (size_t)c->npx * (MOG2_PLANES * 4 + 1);
    else if (c->algo == BGSB_ALGO_DP_ZIVKOVIC_AGMM) *bytes = (size_t)c->npx * ((c->nframes ? c->dpz_K_l : c->gaussians) * 20 + 1);
    else if (c->algo == BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING) *bytes = (size_t)c->npx;
    else if (dp_float_planes(c->algo)) *bytes = (size_t)c->npx * dp_float_planes(c->algo) * 4;
    else if (c->algo == BGSB_ALGO_DP_PRATI_MEDIOD) *bytes = (size_t)c->npx * ((c->nframes ? c->history_size_l : c->history_size) * 5 + 3);
    else if (history_images(c->algo) == 2 || c->algo == BGSB_ALGO_SIGMA_DELTA) *bytes = (size_t)c->npx * 6;
    else *bytes = (size_t)c->npx * 3;
    return BGSB_OK;
}

static int process_batch_impl(bgsb_ctx *c, const uint8_t *d_frames, int T, int w, int h, uint8_t *d_fg,
                              uint8_t *d_bg, int bg_last_only, int *first_fg_valid, int *bg_valid, void *stream,
                              unsigned *d_bits, int bit_thr);

int bgsb_process_batch_dev(bgsb_ctx *c, const uint8_t *d_frames, int T, int w, int h, uint8_t *d_fg,
                           uint8_t *d_bg, int bg_last_only, int *first_fg_valid, int *bg_valid, void *stream)
{
    BGSB_REQUIRE(c && d_frames && d_fg, "null");
    return process_batch_impl(c, d_frames, T, w, h, d_fg, d_bg, bg_last_only, first_fg_valid, bg_valid, stream, nullptr, 0);
}

static int process_batch_impl(bgsb_ctx *c, const uint8_t *d_frames, int T, int w, int h, uint8_t *d_fg,
                              uint8_t *d_bg, int bg_last_only, int *first_fg_valid, int *bg_valid, void *stream,
                              unsigned *d_bits, int bit_thr)
{
    if (int drc = drain(c)) return drc;
    BGSB_REQUIRE(T >= 1, "T >= 1");
    BGSB_CUDA(cudaSetDevice(c->device));
    int rc = ensure_geometry(c, w, h);
    if (rc) return rc;
    rc = order_after_previous(c, (cudaStream_t)stream);
    if (rc) return rc;
    int warm = warmup_frames(c->algo);
    int64_t first = std::max<int64_t>(0, warm - c->nframes);
    if (first_fg_valid) *first_fg_valid = (int)std::min<int64_t>(first, T);
    bool has_bg = writes_background(c->algo);
    // WMM writes its background only from the third frame on (WeightedMovingMeanBGS.cpp:40-51)
    if (bg_valid) *bg_valid = has_bg && d_bg && (first < T);
    if (c->retain_input && ring_history(c->algo) && (T == 1 || c->nstreams == 1)) {
        // "retainInput": the caller keeps the last one (FD) / two (WMV, WMM) frame buffers valid and unmodified, so
        // the history IS those buffers -- as in the host path's upload ring -- and nothing is written back:
        // FD moves its 7 algorithmic bytes per pixel, WMV its 10 (SURVEY 8d).
        if (first < T) {
            rc = launch_range(c, d_frames, T, d_fg, has_bg ? d_bg : nullptr, bg_last_only, false, (cudaStream_t)stream, 0, c->npx);
            if (rc) return rc;
        }
        const size_t fb = (size_t)c->npx * 3;
        const uint8_t *last = d_frames + (size_t)(T - 1) * fb;
        const uint8_t *before = T >= 2 ? d_frames + (size_t)(T - 2) * fb : c->hist_ptr[0];
        c->hist_ptr[1] = before; c->hist_ptr[0] = last;
        c->have_hist = (int)std::min<int64_t>(history_images(c->algo), (int64_t)c->have_hist + T);
        c->nframes += T;
        return BGSB_OK;
    }
    rc = launch_range(c, d_frames, T, d_fg, has_bg ? d_bg : nullptr, bg_last_only, true, (cudaStream_t)stream, 0, c->npx, d_bits, bit_thr);
    if (rc) return rc;
    advance(c, T, true);
    return BGSB_OK;
}

int bgsb_process_dev(bgsb_ctx *c, const uint8_t *d_bgr, int w, int h, uint8_t *d_fg, uint8_t *d_bg,
                     int *fg_valid, int *bg_valid, void *stream)
{
    int first = 0;
    int rc = bgsb_process_batch_dev(c, d_bgr, 1, w, h, d_fg, d_bg, 0, &first, bg_valid, stream);
    if (fg_valid) *fg_valid = (rc == BGSB_OK && first == 0);
    return rc;
}

int bgsb_process(bgsb_ctx *c, const uint8_t *bgr, int w, int h, size_t stride, uint8_t *fg, size_t fg_stride,
                 uint8_t *bg, size_t bg_stride, int *fg_valid, int *bg_valid)
{
    BGSB_REQUIRE(c && bgr && fg, "null");
    BGSB_REQUIRE(stride >= (size_t)w * 3 && fg_stride >= (size_t)w, "stride smaller than a row");
    const size_t bgw = (size_t)w * bg_channels(c ? c->algo : 0);          // bytes per row of img_bgmodel
    BGSB_REQUIRE(!bg || bg_stride >= bgw, "bg stride smaller than a row");
    BGSB_CUDA(cudaSetDevice(c->device));
    int rc = drain(c);
    if (rc) return rc;
    rc = ensure_geometry(c, w, h);
    if (rc) return rc;
    rc = ensure_host_staging(c);
    if (rc) return rc;
    rc = order_after_previous(c, c->stream);
    if (rc) return rc;
    const size_t rows = (size_t)h * c->nstreams;
    const bool fdlike = ring_history(c->algo);
    const int nring = history_images(c->algo) + 1;
    uint8_t *d_in = fdlike ? c->d_ring[c->ring_pos] : c->d_ring[0];
    const int warm = warmup_frames(c->algo);
    const bool out_fg = c->nframes >= warm;
    const bool has_bg = writes_background(c->algo);
    const bool want_bg = has_bg && bg;
    // FD / WMV: history = the previous upload(s) in the ring -- no copy, the frame is read once
    const bool own_hist = !fdlike;

    // Large single frames are cut into row bands (multiples of 32 rows): the upload of band i+1, the
    // kernel on band i and the download of band i-1 overlap on three streams (pixels are independent),
    // so a synchronous IBGS::process costs ~max(H2D, D2H) instead of H2D + kernel + D2H.
    int nchunks = 1, band = h;
    // BGSB_HOST_BANDS=n: the default band count of contexts that did not set "hostBands" (A/B across processes, e.g. under torchrun)
    static const int env_bands = [] { const char *e = getenv("BGSB_HOST_BANDS"); const int v = e ? atoi(e) : 0; return (v >= 1 && v <= 8) ? v : 0; }();
    const int host_bands = c->host_bands_auto ? (env_bands ? env_bands : (want_bg ? 3 : 2)) : c->host_bands;
    if (c->nstreams == 1 && host_bands > 1 && (size_t)w * h * 3 >= (1u << 20) && out_fg && !stencil_algo(c->algo)) {
        band = ((h + host_bands - 1) / host_bands + 31) / 32 * 32;
        if (((size_t)band * w) % MOG2_TILE) band += 32;          // bands start on a state tile
        nchunks = (h + band - 1) / band;
        if (nchunks > 8) { nchunks = 1; band = h; }
    }
    if (nchunks > 1) {
        rc = ensure_pipe_streams(c);
        if (rc) return rc;
    }
    // stage timing (parameter "trace" or BGSB_TRACE=1): events around the uploads, the kernels and the downloads
    const bool tracing = c->trace || trace_env();
    const auto t_wall0 = std::chrono::steady_clock::now();
    nvtxRangePushA(algo_name(c->algo));
    struct NvtxPop { ~NvtxPop() { nvtxRangePop(); } } nvtx_pop;
    if (tracing && !c->ev_t[0]) for (int i = 0; i < 6; i++) BGSB_CUDA(cudaEventCreate(&c->ev_t[i]));
    auto mark = [&](int i, cudaStream_t st) { if (tracing) cudaEventRecord(c->ev_t[i], st); };
    if (nchunks == 1) {
        mark(0, c->stream);
        BGSB_CUDA(copy_rows(d_in, (size_t)w * 3, bgr, stride, (size_t)w * 3, rows, cudaMemcpyHostToDevice, c->stream));
        mark(1, c->stream); mark(2, c->stream);
        if (!out_fg && init_launch_on_warmup(c->algo)) {
            rc = launch_range(c, d_in, 1, c->d_fg, nullptr, 0, own_hist, c->stream, 0, c->npx);
            if (rc) return rc;
        }
        if (out_fg) {
            rc = launch_range(c, d_in, 1, c->d_fg, want_bg ? c->d_bg : nullptr, 0, own_hist, c->stream, 0, c->npx);
            if (rc) return rc;
            mark(3, c->stream); mark(4, c->stream);
            BGSB_CUDA(copy_rows(fg, fg_stride, c->d_fg, (size_t)w, (size_t)w, rows, cudaMemcpyDeviceToHost, c->stream));
            if (want_bg)
                BGSB_CUDA(copy_rows(bg, bg_stride, c->d_bg, bgw, bgw, rows, cudaMemcpyDeviceToHost, c->stream));
        } else { mark(3, c->stream); mark(4, c->stream); }
        mark(5, c->stream);
        BGSB_CUDA(cudaStreamSynchronize(c->stream));
    } else {
        for (int i = 0; i < nchunks; i++) {
            const int r0 = i * band, nr = std::min(band, h - r0);
            const size_t p0 = (size_t)r0 * w;
            if (i == 0) mark(0, c->s_h2d);
            BGSB_CUDA(copy_rows(d_in + p0 * 3, (size_t)w * 3, bgr + (size_t)r0 * stride, stride, (size_t)w * 3, nr,
                                        cudaMemcpyHostToDevice, c->s_h2d));
            BGSB_CUDA(cudaEventRecord(c->ev_up[i], c->s_h2d));
            if (i == nchunks - 1) mark(1, c->s_h2d);
            BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_up[i], 0));
            if (i == 0) mark(2, c->stream);
            rc = launch_range(c, d_in, 1, c->d_fg, want_bg ? c->d_bg : nullptr, 0, own_hist, c->stream, p0, nr * w);
            if (rc) return rc;
            BGSB_CUDA(cudaEventRecord(c->ev_k[i], c->stream));
            if (i == nchunks - 1) mark(3, c->stream);
            BGSB_CUDA(cudaStreamWaitEvent(c->s_d2h, c->ev_k[i], 0));
            if (i == 0) mark(4, c->s_d2h);
            BGSB_CUDA(copy_rows(fg + (size_t)r0 * fg_stride, fg_stride, c->d_fg + p0, (size_t)w, (size_t)w, nr,
                                        cudaMemcpyDeviceToHost, c->s_d2h));
            if (want_bg)
                BGSB_CUDA(copy_rows(bg + (size_t)r0 * bg_stride, bg_stride, c->d_bg + p0 * 3, bgw, bgw, nr,
                                            cudaMemcpyDeviceToHost, c->s_d2h));
        }
        mark(5, c->s_d2h);
        BGSB_CUDA(cudaStreamSynchronize(c->s_d2h));
        BGSB_CUDA(cudaStreamSynchronize(c->stream));
    }
    if (tracing) {
        bgsb_trace &T = c->last_trace;
        float up = 0.f, kn = 0.f, dn = 0.f;
        cudaEventElapsedTime(&up, c->ev_t[0], c->ev_t[1]);
        cudaEventElapsedTime(&kn, c->ev_t[2], c->ev_t[3]);
        cudaEventElapsedTime(&dn, c->ev_t[4], c->ev_t[5]);
        (void)cudaGetLastError();
        T.frame = c->nframes; T.upload_ms = up; T.kernel_ms = kn; T.download_ms = dn; T.bands = nchunks;
        T.wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wall0).count();
        if (trace_env())        // the line FrameProcessor::toc prints (FrameProcessor.cpp:490-494), plus the stage split
            fprintf(stderr, "%s\ttime(sec):%.6f\tupload %.6f kernels %.6f download %.6f (%d band%s, stages overlap)\n", algo_name(c->algo),
                    T.wall_ms * 1e-3, up * 1e-3, kn * 1e-3, dn * 1e-3, nchunks, nchunks > 1 ? "s" : "");
    }
    if (out_fg) advance(c, 1, own_hist);
    else c->nframes += 1;
    if (fdlike) {
        c->hist_ptr[1] = c->hist_ptr[0];
        c->hist_ptr[0] = d_in;
        c->have_hist = std::min(warm, c->have_hist + 1);
        c->ring_pos = (c->ring_pos + 1) % nring;
    }
    if (fg_valid) *fg_valid = out_fg;
    if (bg_valid) *bg_valid = (want_bg && out_fg) ? 1 : 0;
    return BGSB_OK;
}

// Pipelined ingest (SURVEY 8(f) N1, the capture loop VideoCapture.cpp:151-239 / ustc_src/trackingMain.cpp:161-166):
// the same work as bgsb_process, queued.  The call returns as soon as the upload, the kernel and the downloads of this
// frame are enqueued on three streams; the upload of frame t+1 overlaps the download of frame t (PCIe is full duplex),
// which a synchronous IBGS::process cannot do.  The model advances in submission order, so the results are the ones a
// sequence of bgsb_process calls gives.  bgr / fg / bg must stay valid and untouched until bgsb_wait returns, and
// should be page-locked (bgsb_host_alloc) -- pageable buffers work but serialise.  Output slots alternate between two
// device buffers; the kernel of frame t+2 waits for the download of frame t.
int bgsb_submit(bgsb_ctx *c, const uint8_t *bgr, int w, int h, size_t stride, uint8_t *fg, size_t fg_stride,
                uint8_t *bg, size_t bg_stride, int *fg_valid, int *bg_valid)
{
    BGSB_REQUIRE(c && bgr && fg, "null");
    BGSB_REQUIRE(stride >= (size_t)w * 3 && fg_stride >= (size_t)w, "stride smaller than a row");
    const size_t bgw = (size_t)w * bg_channels(c->algo);
    BGSB_REQUIRE(!bg || bg_stride >= bgw, "bg stride smaller than a row");
    BGSB_CUDA(cudaSetDevice(c->device));
    int rc;
    if (c->w != w || c->h != h) {                                  // geometry change: nothing may be in flight
        rc = drain(c);
        if (rc) return rc;
    }
    rc = ensure_geometry(c, w, h);
    if (rc) return rc;
    rc = ensure_host_staging(c);
    if (rc) return rc;
    rc = ensure_pipe_streams(c);
    if (rc) return rc;
    rc = order_after_previous(c, c->stream);
    if (rc) return rc;
    const size_t S = (size_t)c->nstreams;
    {
        cudaError_t e = cudaSuccess;
        if (!c->d_fg2) e = cudaMalloc(&c->d_fg2, S * c->npx);
        if (e == cudaSuccess && !c->d_bg2 && c->d_bg) e = cudaMalloc(&c->d_bg2, S * c->npx * 3);
        if (e != cudaSuccess) { drain(c); return staging_fail(c, e); }
    }
    const size_t rows = (size_t)h * c->nstreams;
    const bool fdlike = ring_history(c->algo);
    const int nring = history_images(c->algo) + 1;
    uint8_t *d_in = fdlike ? c->d_ring[c->ring_pos] : c->d_ring[0];
    const int warm = warmup_frames(c->algo);
    const bool out_fg = c->nframes >= warm;
    const bool want_bg = writes_background(c->algo) && bg;
    const bool own_hist = !fdlike;
    const int slot = (int)(c->seq & 1);
    uint8_t *o_fg = slot ? c->d_fg2 : c->d_fg, *o_bg = slot ? c->d_bg2 : c->d_bg;

    // the input buffer (ring slot) was last read by the previous frame's kernel
    if (c->seq > 0) BGSB_CUDA(cudaStreamWaitEvent(c->s_h2d, c->ev_k[slot ^ 1], 0));
    BGSB_CUDA(copy_rows(d_in, (size_t)w * 3, bgr, stride, (size_t)w * 3, rows, cudaMemcpyHostToDevice, c->s_h2d));
    BGSB_CUDA(cudaEventRecord(c->ev_up[slot], c->s_h2d));
    BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_up[slot], 0));
    if (out_fg || init_launch_on_warmup(c->algo)) {
        BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_dn[slot], 0));       // output slot free (no-op until recorded)
        rc = launch_range(c, d_in, 1, o_fg, (want_bg && out_fg) ? o_bg : nullptr, 0, own_hist, c->stream, 0, c->npx);
        if (rc) return rc;
    }
    BGSB_CUDA(cudaEventRecord(c->ev_k[slot], c->stream));
    if (out_fg) {
        BGSB_CUDA(cudaStreamWaitEvent(c->s_d2h, c->ev_k[slot], 0));
        BGSB_CUDA(copy_rows(fg, fg_stride, o_fg, (size_t)w, (size_t)w, rows, cudaMemcpyDeviceToHost, c->s_d2h));
        if (want_bg) BGSB_CUDA(copy_rows(bg, bg_stride, o_bg, bgw, bgw, rows, cudaMemcpyDeviceToHost, c->s_d2h));
        BGSB_CUDA(cudaEventRecord(c->ev_dn[slot], c->s_d2h));
        advance(c, 1, own_hist);
    } else {
        c->nframes += 1;
    }
    if (fdlike) {
        c->hist_ptr[1] = c->hist_ptr[0];
        c->hist_ptr[0] = d_in;
        c->have_hist = std::min(warm, c->have_hist + 1);
        c->ring_pos = (c->ring_pos + 1) % nring;
    }
    c->seq += 1;
    c->inflight = true;
    if (fg_valid) *fg_valid = out_fg;
    if (bg_valid) *bg_valid = (want_bg && out_fg) ? 1 : 0;
    return BGSB_OK;
}

int bgsb_wait(bgsb_ctx *c)
{
    BGSB_REQUIRE(c, "null ctx");
    return drain(c);
}

int bgsb_process_fanout(bgsb_ctx *const *ctxs, int n, const uint8_t *bgr, int w, int h, size_t stride,
                        uint8_t *const *fg, const size_t *fg_stride, uint8_t *const *bg, const size_t *bg_stride,
                        int *fg_valid, int *bg_valid)
{
    BGSB_REQUIRE(ctxs && bgr && fg && fg_stride && n >= 1 && n <= 16, "bad args");
    BGSB_REQUIRE(stride >= (size_t)w * 3, "stride smaller than a row");
    bgsb_ctx *c0 = ctxs[0];
    for (int k = 0; k < n; k++) { BGSB_REQUIRE(ctxs[k], "null ctx"); if (int drc = drain(ctxs[k])) return drc; }
    for (int k = 0; k < n; k++) {
        BGSB_REQUIRE(ctxs[k] && fg[k], "null context or mask buffer");
        BGSB_REQUIRE(ctxs[k]->device == c0->device && ctxs[k]->nstreams == 1, "fan-out takes single-stream contexts of one device");
        BGSB_REQUIRE(fg_stride[k] >= (size_t)w, "fg stride smaller than a row");
        BGSB_REQUIRE(!(bg && bg[k]) || (bg_stride && bg_stride[k] >= (size_t)w * bg_channels(ctxs[k]->algo)),
                     "bg stride smaller than a row");
        for (int j = 0; j < k; j++) BGSB_REQUIRE(ctxs[j] != ctxs[k], "the same context twice");
    }
    BGSB_CUDA(cudaSetDevice(c0->device));
    for (int k = 0; k < n; k++) {
        int rc = ensure_geometry(ctxs[k], w, h);
        if (rc) return rc;
        rc = ensure_host_staging(ctxs[k]);
        if (rc) return rc;
        rc = ensure_pipe_streams(ctxs[k]);
        if (rc) return rc;
        rc = order_after_previous(ctxs[k], ctxs[k]->stream);
        if (rc) return rc;
    }
    const size_t fbytes = (size_t)w * h * 3;
    if (c0->d_fan_bytes < fbytes) {
        cudaFree(c0->d_fan); c0->d_fan = nullptr; c0->d_fan_bytes = 0;
        BGSB_CUDA(cudaMalloc(&c0->d_fan, fbytes));
        c0->d_fan_bytes = fbytes;
    }
    // row bands as in bgsb_process: the upload of band i+1 overlaps the n kernels on band i (each on its own
    // context's stream) and the downloads of band i-1
    int nchunks = 1, band = h;
    if (c0->host_bands > 1 && fbytes >= (1u << 20)) {
        band = ((h + c0->host_bands - 1) / c0->host_bands + 31) / 32 * 32;
        if (((size_t)band * w) % MOG2_TILE) band += 32;
        nchunks = (h + band - 1) / band;
        if (nchunks > 8) { nchunks = 1; band = h; }
    }
    bool fgv[16], bgv[16];
    for (int k = 0; k < n; k++) {
        bgsb_ctx *c = ctxs[k];
        fgv[k] = c->nframes >= warmup_frames(c->algo);
        bgv[k] = writes_background(c->algo) && bg && bg[k] && fgv[k];
    }
    for (int i = 0; i < nchunks; i++) {
        const int r0 = i * band, nr = std::min(band, h - r0);
        const size_t p0 = (size_t)r0 * w;
        BGSB_CUDA(copy_rows(c0->d_fan + p0 * 3, (size_t)w * 3, bgr + (size_t)r0 * stride, stride, (size_t)w * 3, nr,
                            cudaMemcpyHostToDevice, c0->s_h2d));
        BGSB_CUDA(cudaEventRecord(c0->ev_up[i], c0->s_h2d));
        for (int k = 0; k < n; k++) {
            bgsb_ctx *c = ctxs[k];
            BGSB_CUDA(cudaStreamWaitEvent(c->stream, c0->ev_up[i], 0));
            // a plugin whose mask needs neighbouring pixels (3x3 median) runs once, on the whole frame, after the
            // last band has arrived
            const bool whole = stencil_algo(c->algo);
            if (whole && i != nchunks - 1) continue;
            const size_t q0 = whole ? 0 : p0;
            const int qr0 = whole ? 0 : r0, qnr = whole ? h : nr;
            const size_t bgw = (size_t)w * bg_channels(c->algo);
            // the frame buffer is shared, so every plugin keeps its own history (FD / WMV copy the frame)
            int rc = launch_range(c, c0->d_fan, 1, c->d_fg, writes_background(c->algo) ? c->d_bg : nullptr, 0, true,
                                  c->stream, q0, qnr * w);
            if (rc) return rc;
            BGSB_CUDA(cudaEventRecord(c->ev_k[i], c->stream));
            BGSB_CUDA(cudaStreamWaitEvent(c0->s_d2h, c->ev_k[i], 0));
            if (fgv[k])
                BGSB_CUDA(copy_rows(fg[k] + (size_t)qr0 * fg_stride[k], fg_stride[k], c->d_fg + q0, (size_t)w, (size_t)w, qnr,
                                    cudaMemcpyDeviceToHost, c0->s_d2h));
            if (bgv[k])
                BGSB_CUDA(copy_rows(bg[k] + (size_t)qr0 * bg_stride[k], bg_stride[k], c->d_bg + q0 * 3, bgw, bgw, qnr,
                                    cudaMemcpyDeviceToHost, c0->s_d2h));
        }
    }
    BGSB_CUDA(cudaStreamSynchronize(c0->s_d2h));
    for (int k = 0; k < n; k++) {
        BGSB_CUDA(cudaStreamSynchronize(ctxs[k]->stream));
        advance(ctxs[k], 1, true);
        if (fg_valid) fg_valid[k] = fgv[k];
        if (bg_valid) bg_valid[k] = bgv[k];
    }
    return BGSB_OK;
}

int bgsb_mog2_export_state(bgsb_ctx *c, int si, float *planes, uint8_t *nmodes)
{
    BGSB_REQUIRE(c && planes && nmodes, "null");
    if (int drc = drain(c)) return drc;
    BGSB_REQUIRE(c->algo == BGSB_ALGO_MOG2 && c->d_state, "no MOG2 state");
    BGSB_REQUIRE(si >= 0 && si < c->nstreams, "stream index");
    BGSB_CUDA(cudaSetDevice(c->device));
    BGSB_CUDA(cudaDeviceSynchronize());
    const float *src = c->d_state + (size_t)si * MOG2_PLANES * c->pstride;
    // device tiles [tile][25][64] -> whole-frame planes [25][npx]
    const size_t nt = (size_t)c->npx / MOG2_TILE, rem = (size_t)c->npx % MOG2_TILE;
    for (int q = 0; q < MOG2_PLANES; q++) {
        float *hp = planes + (size_t)q * c->npx;
        if (nt) BGSB_CUDA(cudaMemcpy2D(hp, MOG2_TILE * 4, src + q * MOG2_TILE, MOG2_TILE_FLOATS * 4, MOG2_TILE * 4, nt,
                                       cudaMemcpyDeviceToHost));
        if (rem) BGSB_CUDA(cudaMemcpy(hp + nt * MOG2_TILE, src + nt * MOG2_TILE_FLOATS + q * MOG2_TILE, rem * 4,
                                      cudaMemcpyDeviceToHost));
    }
    BGSB_CUDA(cudaMemcpy(nmodes, c->d_nmodes + (size_t)si * c->pstride, c->npx, cudaMemcpyDeviceToHost));
    if (c->nframes == 0) memset(nmodes, 0, c->npx);
    return BGSB_OK;
}

int bgsb_mog2_import_state(bgsb_ctx *c, int si, int w, int h, int64_t nframes, const float *planes,
                           const uint8_t *nmodes)
{
    BGSB_REQUIRE(c && planes && nmodes, "null");
    if (int drc = drain(c)) return drc;
    BGSB_REQUIRE(c->algo == BGSB_ALGO_MOG2, "not a MOG2 context");
    BGSB_REQUIRE(si >= 0 && si < c->nstreams, "stream index");
    BGSB_REQUIRE(nframes >= 1, "nframes >= 1");
    BGSB_CUDA(cudaSetDevice(c->device));
    int rc = ensure_geometry(c, w, h);
    if (rc) return rc;
    BGSB_CUDA(cudaDeviceSynchronize());
    float *dst = c->d_state + (size_t)si * MOG2_PLANES * c->pstride;
    const size_t nt = (size_t)c->npx / MOG2_TILE, rem = (size_t)c->npx % MOG2_TILE;
    for (int q = 0; q < MOG2_PLANES; q++) {
        const float *hp = planes + (size_t)q * c->npx;
        if (nt) BGSB_CUDA(cudaMemcpy2D(dst + q * MOG2_TILE, MOG2_TILE_FLOATS * 4, hp, MOG2_TILE * 4, MOG2_TILE * 4, nt,
                                       cudaMemcpyHostToDevice));
        if (rem) BGSB_CUDA(cudaMemcpy(dst + nt * MOG2_TILE_FLOATS + q * MOG2_TILE, hp + nt * MOG2_TILE, rem * 4,
                                      cudaMemcpyHostToDevice));
    }
    BGSB_CUDA(cudaMemcpy(c->d_nmodes + (size_t)si * c->pstride, nmodes, c->npx, cudaMemcpyHostToDevice));
    c->nframes = nframes; c->mog2_epoch = 0;
    return BGSB_OK;
}

int bgsb_synth_frames_dev(uint8_t *d_frames, int nstreams, int T, int w, int h, int t0, uint32_t seed0, void *stream)
{
    BGSB_REQUIRE(d_frames && nstreams >= 1 && T >= 1, "bad args");
    return launch_synth(d_frames, nstreams, T, w, h, t0, seed0, (cudaStream_t)stream);
}

// PCIe ceiling of one GPU as this process sees it: page-locked host buffers, two copy streams, no kernels.
int bgsb_copy_probe(int device, size_t bytes_up, size_t bytes_down, int iters, double *sec_up, double *sec_down, double *sec_both)
{
    BGSB_REQUIRE(bytes_up > 0 && bytes_down > 0 && iters >= 1 && sec_up && sec_down && sec_both, "bad args");
    BGSB_CUDA(cudaSetDevice(device));
    void *h_up = nullptr, *h_dn = nullptr, *d_up = nullptr, *d_dn = nullptr;
    // BGSB_PROBE_WC=1: the upload buffer as write-combined memory (what bgsb_host_alloc(.., 1) hands out for input frames)
    static const bool wc = [] { const char *e = getenv("BGSB_PROBE_WC"); return e && e[0] == '1'; }();
    // BGSB_PROBE_SPLIT=k (1..4): each transfer as k pieces on k streams (k copy engines per direction)
    static const int nsplit = [] { const char *e = getenv("BGSB_PROBE_SPLIT"); int k = e ? atoi(e) : 1; return k < 1 ? 1 : (k > 4 ? 4 : k); }();
    cudaStream_t su[4] = {nullptr, nullptr, nullptr, nullptr}, sd[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaError_t e = cudaHostAlloc(&h_up, bytes_up, wc ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaHostAlloc(&h_dn, bytes_down, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaMalloc(&d_up, bytes_up);
    if (e == cudaSuccess) e = cudaMalloc(&d_dn, bytes_down);
    for (int i = 0; i < nsplit && e == cudaSuccess; i++) {
        e = cudaStreamCreateWithFlags(&su[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&sd[i], cudaStreamNonBlocking);
    }
    if (e == cudaSuccess) { memset(h_up, 1, bytes_up); memset(h_dn, 0, bytes_down); }
    auto piece = [&](size_t bytes, int i, size_t *off) { const size_t per = (bytes / nsplit) & ~(size_t)255; *off = per * i; return i == nsplit - 1 ? bytes - per * i : per; };
    auto issue = [&](bool up, bool down) {
        for (int i = 0; i < nsplit && e == cudaSuccess; i++) {
            size_t off = 0, n = 0;
            if (up) { n = piece(bytes_up, i, &off); e = cudaMemcpyAsync((char *)d_up + off, (char *)h_up + off, n, cudaMemcpyHostToDevice, su[i]); }
            if (down && e == cudaSuccess) { n = piece(bytes_down, i, &off); e = cudaMemcpyAsync((char *)h_dn + off, (char *)d_dn + off, n, cudaMemcpyDeviceToHost, sd[i]); }
        }
    };
    auto sync_all = [&]() {
        for (int i = 0; i < nsplit; i++) {
            if (e == cudaSuccess) e = cudaStreamSynchronize(su[i]);
            if (e == cudaSuccess) e = cudaStreamSynchronize(sd[i]);
        }
    };
    auto run = [&](bool up, bool down) -> double {
        for (int w = 0; w < 3; w++) issue(up, down);
        sync_all();
        const auto t0 = std::chrono::steady_clock::now();
        for (int i = 0; i < iters; i++) issue(up, down);
        sync_all();
        return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / iters;
    };
    if (e == cudaSuccess) *sec_up = run(true, false);
    if (e == cudaSuccess) *sec_down = run(false, true);
    if (e == cudaSuccess) *sec_both = run(true, true);
    for (int i = 0; i < 4; i++) { if (su[i]) cudaStreamDestroy(su[i]); if (sd[i]) cudaStreamDestroy(sd[i]); }
    cudaFree(d_up); cudaFree(d_dn);
    if (h_up) cudaFreeHost(h_up);
    if (h_dn) cudaFreeHost(h_dn);
    if (e != cudaSuccess) { set_error("bgsb_copy_probe: %s", cudaGetErrorString(e)); (void)cudaGetLastError(); return BGSB_ERR_CUDA; }
    return BGSB_OK;
}

int bgsb_synth_churn_frames_dev(uint8_t *d_frames, int nstreams, int T, int w, int h, int t0, uint32_t seed0, void *stream)
{
    BGSB_REQUIRE(d_frames && nstreams >= 1 && T >= 1, "bad args");
    return launch_synth_churn(d_frames, nstreams, T, w, h, t0, seed0, (cudaStream_t)stream);
}

}  // extern "C"

namespace bgsb {

bool ctx_can_pack(const bgsb_ctx *c) { return c && c->algo == BGSB_ALGO_MOG2 && c->mog2_variant == 0; }
int ctx_nstreams(const bgsb_ctx *c) { return c->nstreams; }
int ctx_device(const bgsb_ctx *c) { return c->device; }

int ctx_process_frame(bgsb_ctx *c, const uint8_t *d_frames, int w, int h, uint8_t *d_fg, uint8_t *d_bg, unsigned *d_bits,
                      int bit_thr, int *packed, int *fg_valid, int *bg_valid, cudaStream_t stream)
{
    BGSB_REQUIRE(c && d_frames, "null");
    const bool pack = d_bits && ctx_can_pack(c);
    BGSB_REQUIRE(pack || d_fg, "this plugin needs a byte mask buffer");
    if (packed) *packed = pack;
    int first = 0;
    int rc = process_batch_impl(c, d_frames, 1, w, h, d_fg, d_bg, 0, &first, bg_valid, (void *)stream, pack ? d_bits : nullptr, bit_thr);
    if (fg_valid) *fg_valid = (rc == BGSB_OK && first == 0);
    return rc;
}

}  // namespace bgsb
