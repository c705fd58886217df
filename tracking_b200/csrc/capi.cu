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
#include <string>
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

// What the host code knows about each plugin: one row per algorithm id of include/bgsb200.h.
enum Family { FAM_SIMPLE, FAM_MOG2, FAM_DPZ, FAM_DPS, FAM_SD, FAM_PRATI, FAM_ASBL };   // how launch_range runs it
enum Model {
    MODEL_BYTES,      // `count` images of 3 bytes per pixel (d_hist)
    MODEL_MIXTURE,    // per-pixel mixture of `count` modes (0: "gaussians") in the MOG2 tile layout (d_state / d_nmodes)
    MODEL_DP_PLANES,  // `count` fp32 planes per pixel (d_state, [S][planes][pstride])
    MODEL_PRATI,      // the medoid ring block (d_prati), sized by "historySize" on the first frame (launch_range)
};
struct PluginInfo {
    int id;
    const char *name;
    Family family;
    int warmup;              // frames before the first mask (SigmaDeltaBGS.cpp:28-33; WMM's background too, .cpp:40-51)
    bool warmup_launch;      // a warm-up frame still needs a kernel: the model is initialised from it
    bool ring_history;       // the history is the previous input frame(s): on the host path it lives in the upload ring
    int history;             // history images the plugin keeps (have_hist saturates there)
    Model model;
    int count;               // byte images or fp32 planes of the model
    int bg_channels;         // channels of img_bgmodel
    bool stencil;            // the mask depends on neighbouring pixels: whole frames only, no row bands
    bool writes_bg;          // ever writes img_bgmodel
    bool real_threshold;     // "threshold" reads back as the real value set (else as the int member)
    // loadConfig defaults
    double alpha, threshold;
    int sampling_rate, learning_frames;
};
// Byte images: FD the previous frame, WMV / WMM the two previous ones, ABL / StaticFD the 8-bit background, ASBL the gray
// model (AdaptiveSelectiveBackgroundLearning.cpp:103) and scratch, SigmaDelta Mt and Vt, DPAdaptiveMedian the median.
// Stencils: ASBL's 3x3 median, DPPratiMediod's hysteresis over the 8 neighbours.  loadConfig defaults: ASBL .cpp:121-125,
// DPZivkovicAGMMBGS.cpp:97-100, DPAdaptiveMedianBGS.cpp:101-103, DPMeanBGS.cpp:103-105, DPWrenGABGS.cpp:103-105 (float
// literals read into doubles), DPPratiMediodBGS.cpp:104-107.
static const PluginInfo PLUGINS[] = {
    // id, name, family, warmup, warmup_launch, ring_history, history, model, count, bg_channels, stencil, writes_bg, real_threshold, alpha, threshold, sampling_rate, learning_frames
    {BGSB_ALGO_FRAME_DIFFERENCE, "FrameDifferenceBGS", FAM_SIMPLE, 1, false, true, 1, MODEL_BYTES, 1, 3, false, false, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_STATIC_FRAME_DIFFERENCE, "StaticFrameDifferenceBGS", FAM_SIMPLE, 0, false, false, 1, MODEL_BYTES, 1, 3, false, true, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_WEIGHTED_MOVING_MEAN, "WeightedMovingMeanBGS", FAM_SIMPLE, 2, false, true, 2, MODEL_BYTES, 2, 3, false, true, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_WEIGHTED_MOVING_VARIANCE, "WeightedMovingVarianceBGS", FAM_SIMPLE, 2, false, true, 2, MODEL_BYTES, 2, 3, false, false, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_MOG2, "MixtureOfGaussianV2BGS", FAM_MOG2, 0, false, false, 0, MODEL_MIXTURE, MOG2_K, 3, false, true, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_ADAPTIVE_BG_LEARNING, "AdaptiveBackgroundLearning", FAM_SIMPLE, 0, false, false, 1, MODEL_BYTES, 1, 3, false, true, false, 0.05, 15, 7, 90},
    {BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING, "AdaptiveSelectiveBackgroundLearning", FAM_ASBL, 0, false, false, 1, MODEL_BYTES, 2, 1, true, true, false, 0.05, 25, 7, 90},
    {BGSB_ALGO_DP_ADAPTIVE_MEDIAN, "DPAdaptiveMedianBGS", FAM_DPS, 0, false, false, 1, MODEL_BYTES, 1, 3, false, false, false, 0.05, 40, 7, 30},
    {BGSB_ALGO_DP_ZIVKOVIC_AGMM, "DPZivkovicAGMMBGS", FAM_DPZ, 0, false, false, 0, MODEL_MIXTURE, 0, 3, false, false, true, 0.001, 25, 7, 90},
    {BGSB_ALGO_DP_MEAN, "DPMeanBGS", FAM_DPS, 0, false, false, 0, MODEL_DP_PLANES, 3, 3, false, false, false, (double)1e-6f, 2700, 7, 30},
    {BGSB_ALGO_DP_WREN_GA, "DPWrenGABGS", FAM_DPS, 0, false, false, 0, MODEL_DP_PLANES, 4, 3, false, false, true, (double)0.005f, (double)12.25f, 7, 30},
    {BGSB_ALGO_DP_PRATI_MEDIOD, "DPPratiMediodBGS", FAM_PRATI, 0, false, false, 0, MODEL_PRATI, 0, 3, true, false, false, 0.05, 30, 5, 90},
    {BGSB_ALGO_SIGMA_DELTA, "SigmaDeltaBGS", FAM_SD, 1, true, false, 1, MODEL_BYTES, 2, 3, false, false, false, 0.05, 15, 7, 90},
};

static const PluginInfo *plugin_info(int algo)
{
    for (const PluginInfo &p : PLUGINS)
        if (p.id == algo) return &p;
    return nullptr;
}

struct bgsb_ctx {
    int algo = 0, device = 0, nstreams = 1;
    const PluginInfo *pi = nullptr;
    // plugin parameters (XML keys of the reference); alpha, threshold (thr / dpz_threshold), samplingRate and
    // learningFrames are set from the plugin's loadConfig defaults at create (PLUGINS)
    double alpha = 0;
    int limit = -1;
    int enable_thr = 1, thr = 0, enable_weight = 1, gray_variant = 0;
    // cv::BackgroundSubtractorMOG2 defaults (SURVEY 8a row a6)
    int history = 500;
    float Tb = 16.f, Tg = 9.f, TB = 0.9f, varInit = 15.f, varMin = 4.f, varMax = 75.f, CT = 0.05f, tau = 0.5f;
    int detect_shadows = 1, shadow_value = 127;
    bool host_bands_auto = true;   // "hostBands" not set: 3 bands when the background image goes back too, else 2 (1080p MOG2: 266 vs 274 us with the image, 176 vs 177 without; 4 bands 279 / 185)
    int host_bands = 2;        // row bands of the host-path upload/compute/download pipeline (1 = no overlap); 2 measured best at 1080p (277 vs 289 us with 4: each band costs ~8 host API calls)
    // AdaptiveSelectiveBackgroundLearning (defaults of its loadConfig, .cpp:121-125)
    int learning_frames = 0, asbl_counter = 0;
    int asbl_cur = 0;          // which of the two ASBL model buffers holds the model
    double alpha_learn = 0.05, alpha_detection = 0.05;
    // DPZivkovicAGMMBGS: "threshold" as a real number, "gaussians" (defaults of its loadConfig, DPZivkovicAGMMBGS.cpp:97-100)
    double dpz_threshold = 0;
    int gaussians = 3;
    // ... which the reference hands to the model ONCE, on the first frame (DPZivkovicAGMMBGS.cpp:58-65): later changes
    // of threshold / alpha / gaussians have no effect until the model is reset.  Latched copies used by the kernel:
    double dpz_thr_l = 25.0, dpz_alpha_l = 0.001;
    int dpz_K_l = 3;
    // DPAdaptiveMedianBGS / DPMeanBGS / DPWrenGABGS: "threshold" (kept in dpz_threshold), "alpha", "samplingRate",
    // "learningFrames"; handed to the model once, on the first frame, like DPZivkovic's (latched in dpz_thr_l / dpz_alpha_l)
    int sampling_rate = 0, sampling_rate_l = 7;
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
    int mog2_variant = 0;      // see launch_mog2 (mog2.cu): 0 production, 1 straight restatement
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
    // "inputFormat": BGR, or YUV 4:2:0 frames (NV12 / I420) that ingest/yuv420.cu converts to BGR before the plugin runs;
    // the model and the history stay BGR, so the format may change between calls
    int input_format = BGSB_INPUT_BGR;
    uint8_t *d_yuv = nullptr;             // host paths: the uploaded YUV frames [S][3h/2][w] (fan-out: the first context's)
    uint8_t *d_conv = nullptr;            // device paths: the converted frames [S][T][h][w][3]
    size_t d_conv_bytes = 0;
    // "gaussianBlur": the reference PreProcessor's cv::GaussianBlur(Size(7, 7), 1.5), which prep/gauss7.cu applies to
    // every BGR frame (after the YUV conversion) before the plugin sees it; the history is the blurred frame
    int gaussian_blur = 0;
    uint8_t *d_prep = nullptr;            // host paths: the BGR frames before the blur [S][h][w][3] (fan-out: the first context's)
    uint8_t *d_blur = nullptr;            // device paths: the blurred frames [S][T][h][w][3]
    size_t d_blur_bytes = 0;
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

static bool trace_env()
{
    static const bool on = [] { const char *e = getenv("BGSB_TRACE"); return e && e[0] && e[0] != '0'; }();
    return on;
}

// Staging buffers of the host paths.
static void free_staging(bgsb_ctx *c)
{
    for (int i = 0; i < 3; i++) { cudaFree(c->d_ring[i]); c->d_ring[i] = nullptr; }
    cudaFree(c->d_fg); c->d_fg = nullptr;
    cudaFree(c->d_bg); c->d_bg = nullptr;
    cudaFree(c->d_fg2); c->d_fg2 = nullptr;
    cudaFree(c->d_bg2); c->d_bg2 = nullptr;
    cudaFree(c->d_yuv); c->d_yuv = nullptr;
    cudaFree(c->d_prep); c->d_prep = nullptr;
}

static void free_buffers(bgsb_ctx *c)
{
    cudaFree(c->d_state); c->d_state = nullptr;
    cudaFree(c->d_nmodes); c->d_nmodes = nullptr;
    cudaFree(c->d_abl_lut); c->d_abl_lut = nullptr; c->lut_alpha = -1.;
    for (int i = 0; i < 2; i++) { cudaFree(c->d_hist[i]); c->d_hist[i] = nullptr; c->hist_ptr[i] = nullptr; }
    free_staging(c);
    cudaFree(c->d_fan); c->d_fan = nullptr; c->d_fan_bytes = 0;
    cudaFree(c->d_conv); c->d_conv = nullptr; c->d_conv_bytes = 0;
    cudaFree(c->d_blur); c->d_blur = nullptr; c->d_blur_bytes = 0;
    cudaFree(c->d_prati); c->d_prati = nullptr; c->prati_bytes = 0; c->prati_n = c->prati_pos = 0;
    c->w = c->h = c->npx = 0; c->pstride = 0;
    c->nframes = 0; c->mog2_epoch = 0; c->have_hist = 0; c->ring_pos = 0;
}

// (Re)allocate model state for a geometry.  The reference discovers the frame size on the first
// process() call; cv::BackgroundSubtractorMOG2::operator() re-initialises when it changes.
static int ensure_geometry(bgsb_ctx *c, int w, int h)
{
    if (c->w == w && c->h == h) return BGSB_OK;
    const PluginInfo &P = *c->pi;
    BGSB_REQUIRE(w > 0 && h > 0, "empty frame");
    BGSB_REQUIRE((long long)w * h < (1LL << 30), "frame too large");
    BGSB_REQUIRE(P.model != MODEL_MIXTURE || (long long)w * h <= (1LL << 27), "mixture-model frames are limited to 2^27 pixels");
    free_buffers(c);                              // geometry fields are 0 from here until every allocation has succeeded
    const int npx = w * h;
    const size_t pstride = ((size_t)npx + MOG2_TILE - 1) / MOG2_TILE * MOG2_TILE;       // whole state tiles
    const size_t S = (size_t)c->nstreams;
    cudaError_t e = cudaSuccess;
    switch (P.model) {
    case MODEL_MIXTURE: {
        const size_t fb = S * MOG2_PLANES * pstride * sizeof(float);
        e = cudaMalloc(&c->d_state, fb);
        if (e == cudaSuccess) e = cudaMalloc(&c->d_nmodes, S * pstride);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_state, 0, fb, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->d_nmodes, 0, S * pstride, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        break;
    }
    case MODEL_DP_PLANES:
        e = cudaMalloc(&c->d_state, S * P.count * pstride * sizeof(float));      // written in full by the first frame
        break;
    case MODEL_PRATI:
        break;
    case MODEL_BYTES:
        for (int i = 0; i < P.count && e == cudaSuccess; i++) e = cudaMalloc(&c->d_hist[i], S * npx * 3);
        break;
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

// All-or-nothing like ensure_geometry.
static int staging_fail(bgsb_ctx *c, cudaError_t e)
{
    set_error("host staging (%d x %d x %d streams): %s", c->w, c->h, c->nstreams, cudaGetErrorString(e));
    (void)cudaGetLastError();
    free_staging(c);
    return BGSB_ERR_CUDA;
}

static int ensure_host_staging(bgsb_ctx *c)
{
    const PluginInfo &P = *c->pi;
    const size_t S = (size_t)c->nstreams;
    cudaError_t e = cudaSuccess;
    if (!c->d_ring[0]) {
        const int nr = P.ring_history ? P.history + 1 : 1;
        for (int i = 0; i < nr && e == cudaSuccess; i++) e = cudaMalloc(&c->d_ring[i], S * c->npx * 3);
        c->ring_pos = 0;
    }
    if (e == cudaSuccess && !c->d_fg) e = cudaMalloc(&c->d_fg, S * c->npx);
    if (e == cudaSuccess && !c->d_bg && P.writes_bg) e = cudaMalloc(&c->d_bg, S * c->npx * 3);
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

// ---- YUV 4:2:0 input -------------------------------------------------------------------------------
// The layout cv::cvtColor(COLOR_YUV2BGR_NV12 / _I420) reads: one 8-bit image of 3h/2 rows of w bytes.  NV12: h Y rows,
// then h/2 rows of interleaved U,V; I420: the Y plane, the U plane (w/2 x h/2), the V plane, densely packed.  Host
// frames have `stride` bytes between rows (I420: stride == w); device frames are dense, [frames][3h/2][w].
static int check_yuv_frame(int fmt, int w, int h, size_t stride)
{
    BGSB_REQUIRE(w > 0 && h > 0 && w % 2 == 0 && h % 2 == 0, "YUV 4:2:0 input (inputFormat NV12 / I420) needs an even width and height");
    BGSB_REQUIRE(stride >= (size_t)w, "stride smaller than a row");
    BGSB_REQUIRE(fmt != BGSB_INPUT_I420 || stride == (size_t)w, "I420 frames are dense planes: stride must equal w");
    return BGSB_OK;
}

// Rows [r0, r0 + nr) (r0, nr even) of `nframes` dense device YUV frames at src -> the same rows of dense BGR frames at dst.
static int convert_yuv(int fmt, const uint8_t *src, int w, int h, int r0, int nr, int nframes, uint8_t *dst, cudaStream_t st)
{
    const size_t W = (size_t)w, H = (size_t)h;
    Yuv420Launch L;
    memset(&L, 0, sizeof(L));
    L.y = src + r0 * W; L.y_pitch = W;
    if (fmt == BGSB_INPUT_NV12) {
        L.u = src + (H + r0 / 2) * W; L.c_pitch = W;
    } else {
        L.u = src + H * W + (r0 / 2) * (W / 2); L.v = L.u + (H / 2) * (W / 2); L.c_pitch = W / 2; L.planar = 1;
    }
    L.src_frame_stride = H * W * 3 / 2;
    L.bgr = dst + r0 * W * 3; L.dst_frame_stride = H * W * 3;
    L.w = w; L.rows = nr; L.nframes = nframes;
    return launch_yuv420_to_bgr(L, st);
}

// Host rows [r0, r0 + nr) of `nframes` YUV frames stacked `stride`-apart rows -> the dense device staging at dst.  A band
// (r0, nr) != (0, h) is one frame's Y rows and chroma rows; I420's planes are dense, so each plane's band is one span.
static cudaError_t upload_yuv(int fmt, uint8_t *dst, const uint8_t *src, size_t stride, int w, int h, int r0, int nr,
                              int nframes, cudaStream_t st)
{
    const size_t W = (size_t)w, H = (size_t)h;
    if (r0 == 0 && nr == h) return copy_rows(dst, W, src, stride, W, (size_t)nframes * H * 3 / 2, cudaMemcpyHostToDevice, st);
    cudaError_t e = copy_rows(dst + r0 * W, W, src + r0 * stride, stride, W, nr, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    if (fmt == BGSB_INPUT_NV12)
        return copy_rows(dst + (H + r0 / 2) * W, W, src + (H + r0 / 2) * stride, stride, W, nr / 2, cudaMemcpyHostToDevice, st);
    const size_t q = W / 2, off = H * W + (r0 / 2) * q, n = (nr / 2) * q;
    e = cudaMemcpyAsync(dst + off, src + off, n, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    return cudaMemcpyAsync(dst + off + (H / 2) * q, src + off + (H / 2) * q, n, cudaMemcpyHostToDevice, st);
}

static int ensure_yuv_staging(bgsb_ctx *c)
{
    if (c->d_yuv) return BGSB_OK;
    const cudaError_t e = cudaMalloc(&c->d_yuv, (size_t)c->nstreams * c->npx * 3 / 2);
    if (e != cudaSuccess) return staging_fail(c, e);
    return BGSB_OK;
}

// ---- "gaussianBlur" --------------------------------------------------------------------------------
// Output rows [r0, r0 + nr) of `nframes` dense BGR frames at src -> the same rows at dst.  Rows up to 3 beyond the band
// are read, so on the host paths band i is blurred only once band i + 1 has arrived.
static int blur_frames(const uint8_t *src, int w, int h, int r0, int nr, int nframes, uint8_t *dst, cudaStream_t st)
{
    Gauss7Launch L;
    memset(&L, 0, sizeof(L));
    L.src = src; L.dst = dst; L.frame_stride = (size_t)w * h * 3;
    L.w = w; L.h = h; L.r0 = r0; L.nr = nr; L.nframes = nframes;
    return launch_gauss7(L, st);
}

// host paths with the blur: the uploaded (or converted) BGR frames land here and are blurred into the ring slot
static int ensure_prep_staging(bgsb_ctx *c)
{
    if (c->d_prep) return BGSB_OK;
    const cudaError_t e = cudaMalloc(&c->d_prep, (size_t)c->nstreams * c->npx * 3);
    if (e != cudaSuccess) return staging_fail(c, e);
    return BGSB_OK;
}

// Launch the kernels that advance the model by T frames that sit in device memory, for pixels [p0, p0+pcount) of the
// frame(s); p0 must be a multiple of 64 (a MOG2 state tile).  A sub-range is only used for single-stream, single-frame
// calls (host-path row bands), so everything that happens once per call lives in latch_first_frame and advance.
// `own_history`: write FD/WMV history into the context's own buffers (caller's frame buffers may be reused after the call).
static int launch_range(bgsb_ctx *c, const uint8_t *d_frames, int T, uint8_t *d_fg, uint8_t *d_bg,
                        int bg_last_only, bool own_history, cudaStream_t stream, size_t p0, int pcount,
                        unsigned *d_bits = nullptr, int bit_thr = 0)
{
    switch (c->pi->family) {
    case FAM_MOG2: {
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
        break;
    }
    case FAM_DPZ:
        for (int t = 0; t < T; t++) {
            DpzLaunch L;
            memset(&L, 0, sizeof(L));
            // batch layouts: frames [S][T][npx*3], masks [S][T][npx]; pixels [p0, p0+pcount), p0 on a state tile
            L.frame = d_frames + ((size_t)t * c->npx + p0) * 3; L.frame_stride = (size_t)T * c->npx * 3;
            L.fg = d_fg + (size_t)t * c->npx + p0; L.fg_stride = (size_t)T * c->npx;
            L.state = c->d_state + p0 * MOG2_PLANES; L.nmodes = c->d_nmodes + p0; L.pstride = c->pstride;
            L.npx = pcount; L.K = c->dpz_K_l;
            L.fresh = (c->nframes + t == 0);
            L.low_thr = (float)c->dpz_thr_l; L.alpha = (float)c->dpz_alpha_l;
            int rc = launch_dpz(L, c->nstreams, stream);
            if (rc) return rc;
        }
        break;
    case FAM_DPS:
        for (int t = 0; t < T; t++) {
            DpsLaunch L;
            memset(&L, 0, sizeof(L));
            const int64_t frame_num = c->nframes + t;                      // the wrappers' frameNumber
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
        break;
    case FAM_SD:
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
        break;
    case FAM_PRATI:
        BGSB_REQUIRE(p0 == 0 && pcount == c->npx, "DPPratiMediod works on whole frames (8-neighbour hysteresis)");
        for (int t = 0; t < T; t++) {
            const int64_t frame_num = c->nframes + t;                      // the wrapper's frameNumber
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
        break;
    case FAM_ASBL: {
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
        break;
    }
    case FAM_SIMPLE: {
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
        break;
    }
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

// The reference hands threshold, alpha, gaussians, samplingRate and historySize to its model once, on the first frame
// (DPZivkovicAGMMBGS.cpp:58-65, DPPratiMediodBGS.cpp:57-62): later changes have no effect until the model is reset.
// Each plugin reads only its own latched fields.  Called once per call, before its first launch.
static void latch_first_frame(bgsb_ctx *c)
{
    if (c->nframes != 0) return;
    c->dpz_thr_l = c->dpz_threshold; c->dpz_alpha_l = c->alpha; c->dpz_K_l = c->gaussians;
    c->sampling_rate_l = c->sampling_rate; c->history_size_l = c->history_size;
    c->prati_n = 0; c->prati_pos = 0;
}

// Bookkeeping once per call, after its T frames went through launch_range.
static void advance(bgsb_ctx *c, int T, bool own_history)
{
    if (own_history) {
        c->have_hist = (int)std::min<int64_t>(c->pi->history, (int64_t)c->have_hist + T);
        c->hist_ptr[0] = c->d_hist[0]; c->hist_ptr[1] = c->d_hist[1];
    }
    if (c->pi->family == FAM_MOG2 && c->alpha >= 1) c->mog2_epoch = c->nframes + T - 1;  // the last frame re-initialised the model
    c->nframes += T;
}

// FD / WMV / WMM: the frame at d_in, which stays valid until the next call, becomes the newest history image; the
// host paths upload the next frame into the following ring slot.
static void remember_input(bgsb_ctx *c, const uint8_t *d_in)
{
    c->hist_ptr[1] = c->hist_ptr[0];
    c->hist_ptr[0] = d_in;
    c->have_hist = std::min(c->pi->history, c->have_hist + 1);
    c->ring_pos = (c->ring_pos + 1) % (c->pi->history + 1);
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

// Arguments of bgsb_process / bgsb_submit: one frame, or a group's frames stacked.
static int check_host_frame(const bgsb_ctx *c, const uint8_t *bgr, int w, int h, size_t stride, const uint8_t *fg,
                            size_t fg_stride, const uint8_t *bg, size_t bg_stride)
{
    BGSB_REQUIRE(c && bgr && fg, "null");
    if (c->input_format != BGSB_INPUT_BGR) {
        int rc = check_yuv_frame(c->input_format, w, h, stride);
        if (rc) return rc;
    }
    BGSB_REQUIRE(stride >= (size_t)w * (c->input_format == BGSB_INPUT_BGR ? 3 : 1) && fg_stride >= (size_t)w, "stride smaller than a row");
    BGSB_REQUIRE(!bg || bg_stride >= (size_t)w * c->pi->bg_channels, "bg stride smaller than a row");
    return BGSB_OK;
}

// Set-up of a host-buffer call on the context's own stream, after the model has been drained where needed.
static int host_setup(bgsb_ctx *c, int w, int h)
{
    int rc = ensure_geometry(c, w, h);
    if (!rc) rc = ensure_host_staging(c);
    if (!rc) rc = ensure_pipe_streams(c);
    if (!rc) rc = order_after_previous(c, c->stream);
    if (!rc) latch_first_frame(c);
    return rc;
}

// A host-buffer frame returns its mask once the warm-up is over, and then its background image if one is asked for
// and the plugin writes one.
static bool mask_due(const bgsb_ctx *c) { return c->nframes >= c->pi->warmup; }
static bool bg_due(const bgsb_ctx *c, const uint8_t *bg) { return bg && c->pi->writes_bg && mask_due(c); }

// Row bands of the host-path pipeline: the upload of band i+1, the kernels on band i and the download of band i-1
// overlap on three streams (pixels are independent), so a synchronous call costs ~max(H2D, D2H) instead of
// H2D + kernel + D2H.  Bands are multiples of 32 rows that start on a state tile; frames under 1 MB, and cuts into
// more than 8 bands, stay whole.
struct Bands { int n, rows; };
static Bands plan_bands(int w, int h, int bands)
{
    if (bands <= 1 || (size_t)w * h * 3 < (1u << 20)) return {1, h};
    int band = ((h + bands - 1) / bands + 31) / 32 * 32;
    if (((size_t)band * w) % MOG2_TILE) band += 32;
    const int n = (h + band - 1) / band;
    return n > 8 ? Bands{1, h} : Bands{n, band};
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
    const PluginInfo *pi = plugin_info(algo);
    if (!pi) {
        std::string ids;
        for (const PluginInfo &p : PLUGINS) ids += (ids.empty() ? "" : ", ") + std::to_string(p.id) + " " + p.name;
        set_error("unknown algorithm id %d (USTC_BGS ids: %s)", algo, ids.c_str());
        return BGSB_ERR_ARG;
    }
    BGSB_REQUIRE(nstreams >= 1 && nstreams <= 65535, "nstreams out of range");
    BGSB_CUDA(cudaSetDevice(device));
    bgsb_ctx *c = new bgsb_ctx();
    c->algo = algo; c->pi = pi; c->device = device; c->nstreams = nstreams;
    c->alpha = pi->alpha; c->thr = (int)pi->threshold; c->dpz_threshold = pi->threshold;
    c->sampling_rate = pi->sampling_rate; c->learning_frames = pi->learning_frames;
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
    else if (k == "retainInput") {
        BGSB_REQUIRE(v == 0 || c->input_format == BGSB_INPUT_BGR, "retainInput cannot be combined with a YUV inputFormat: the "
                     "converted frames are the library's, so the caller's buffers cannot serve as the history");
        BGSB_REQUIRE(v == 0 || !c->gaussian_blur, "retainInput cannot be combined with gaussianBlur: the history is the "
                     "blurred frame, so the caller's unblurred buffers cannot serve as it");
        c->retain_input = (v != 0);
    }
    else if (k == "gaussianBlur") {
        BGSB_REQUIRE(v == 0 || v == 1, "gaussianBlur is 0 or 1");
        BGSB_REQUIRE(v == 0 || !c->retain_input, "gaussianBlur cannot be combined with retainInput: the history is the "
                     "blurred frame, so the caller's unblurred buffers cannot serve as it");
        c->gaussian_blur = (int)v;
    }
    else if (k == "inputFormat") {
        BGSB_REQUIRE(v == BGSB_INPUT_BGR || v == BGSB_INPUT_NV12 || v == BGSB_INPUT_I420,
                     "inputFormat is 0 (BGSB_INPUT_BGR), 1 (BGSB_INPUT_NV12) or 2 (BGSB_INPUT_I420)");
        BGSB_REQUIRE(v == BGSB_INPUT_BGR || !c->retain_input, "a YUV inputFormat cannot be combined with retainInput: the "
                     "converted frames are the library's, so the caller's buffers cannot serve as the history");
        c->input_format = (int)v;
    }
    else if (k == "quietGroups") c->wmv_quiet = (v != 0);
    else if (k == "trace") c->trace = (v != 0);
    else if (k == "kernelVariant") { BGSB_REQUIRE(v == 0 || v == 1, "kernelVariant is 0 or 1"); c->mog2_variant = (int)v; }
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
    else if (k == "threshold") *v = c->pi->real_threshold ? c->dpz_threshold : c->thr;
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
    else if (k == "inputFormat") *v = c->input_format;
    else if (k == "gaussianBlur") *v = c->gaussian_blur;
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
    const PluginInfo &P = *c->pi;
    const size_t npx = (size_t)c->npx;
    switch (P.model) {
    case MODEL_MIXTURE: {     // fp32 weight, variance and 3 means per mode, and the mode count; DPZivkovic: "gaussians" modes
        const int K = P.count ? P.count : (c->nframes ? c->dpz_K_l : c->gaussians);
        *bytes = npx * (K * 5 * 4 + 1);
        break;
    }
    case MODEL_DP_PLANES: *bytes = npx * P.count * 4; break;
    case MODEL_PRATI: *bytes = npx * ((c->nframes ? c->history_size_l : c->history_size) * 5 + 3); break;
    case MODEL_BYTES: *bytes = npx * (P.family == FAM_ASBL ? 1 : P.count * 3); break;    // ASBL: the gray model; image 1 is scratch
    }
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
    const bool yuv = c->input_format != BGSB_INPUT_BGR;
    if (yuv) {
        int rc = check_yuv_frame(c->input_format, w, h, (size_t)w);
        if (rc) return rc;
    }
    BGSB_CUDA(cudaSetDevice(c->device));
    int rc = ensure_geometry(c, w, h);
    if (rc) return rc;
    rc = order_after_previous(c, (cudaStream_t)stream);
    if (rc) return rc;
    latch_first_frame(c);
    if (yuv) {
        // the caller's YUV frames become BGR frames in a library-owned scratch, on the caller's stream; the plugin then
        // runs on the scratch exactly as on BGR frames, writing its history back (the scratch is reused by the next call)
        const size_t need = (size_t)c->nstreams * T * c->npx * 3;
        if (c->d_conv_bytes < need) {
            cudaFree(c->d_conv); c->d_conv = nullptr; c->d_conv_bytes = 0;
            BGSB_CUDA(cudaMalloc(&c->d_conv, need));
            c->d_conv_bytes = need;
        }
        rc = convert_yuv(c->input_format, d_frames, w, h, 0, h, c->nstreams * T, c->d_conv, (cudaStream_t)stream);
        if (rc) return rc;
        d_frames = c->d_conv;
    }
    const bool blur = c->gaussian_blur != 0;
    if (blur) {          // likewise: all S x T frames blurred in one launch into a second scratch
        const size_t need = (size_t)c->nstreams * T * c->npx * 3;
        if (c->d_blur_bytes < need) {
            cudaFree(c->d_blur); c->d_blur = nullptr; c->d_blur_bytes = 0;
            BGSB_CUDA(cudaMalloc(&c->d_blur, need));
            c->d_blur_bytes = need;
        }
        rc = blur_frames(d_frames, w, h, 0, h, c->nstreams * T, c->d_blur, (cudaStream_t)stream);
        if (rc) return rc;
        d_frames = c->d_blur;
    }
    int64_t first = std::max<int64_t>(0, c->pi->warmup - c->nframes);
    if (first_fg_valid) *first_fg_valid = (int)std::min<int64_t>(first, T);
    const bool has_bg = c->pi->writes_bg;
    if (bg_valid) *bg_valid = has_bg && d_bg && (first < T);
    if (c->retain_input && !yuv && !blur && c->pi->ring_history && (T == 1 || c->nstreams == 1)) {
        // "retainInput": the caller keeps the last one (FD) / two (WMV, WMM) frame buffers valid and unmodified, so
        // the history IS those buffers -- as in the host path's upload ring -- and nothing is written back:
        // FD moves its 7 algorithmic bytes per pixel, WMV its 10 (SURVEY 8d).
        if (first < T) {
            rc = launch_range(c, d_frames, T, d_fg, has_bg ? d_bg : nullptr, bg_last_only, false, (cudaStream_t)stream, 0, c->npx);
            if (rc) return rc;
        }
        const size_t fb = (size_t)c->npx * 3;
        if (T >= 2) remember_input(c, d_frames + (size_t)(T - 2) * fb);
        remember_input(c, d_frames + (size_t)(T - 1) * fb);
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
    int rc = check_host_frame(c, bgr, w, h, stride, fg, fg_stride, bg, bg_stride);
    if (rc) return rc;
    BGSB_CUDA(cudaSetDevice(c->device));
    rc = drain(c);
    if (rc) return rc;
    rc = host_setup(c, w, h);
    if (rc) return rc;
    const PluginInfo &P = *c->pi;
    const size_t rows = (size_t)h * c->nstreams;
    const size_t bgw = (size_t)w * P.bg_channels;         // bytes per row of img_bgmodel
    uint8_t *d_in = c->d_ring[c->ring_pos];
    const int fmt = c->input_format;       // YUV: the upload lands in d_yuv and is converted into the ring slot
    if (fmt != BGSB_INPUT_BGR && (rc = ensure_yuv_staging(c))) return rc;
    const bool blur = c->gaussian_blur != 0;   // blur: the BGR frame lands in d_prep and is blurred into the ring slot
    if (blur && (rc = ensure_prep_staging(c))) return rc;
    uint8_t *const d_up = blur ? c->d_prep : d_in;
    const bool out_fg = mask_due(c), want_bg = bg_due(c, bg);
    // FD / WMV: history = the previous upload(s) in the ring -- no copy, the frame is read once
    const bool own_hist = !P.ring_history;
    const int host_bands = c->host_bands_auto ? (want_bg ? 3 : 2) : c->host_bands;
    const Bands B = plan_bands(w, h, (c->nstreams == 1 && out_fg && !P.stencil) ? host_bands : 1);
    const int nchunks = B.n, band = B.rows;
    // stage timing (parameter "trace" or BGSB_TRACE=1): events around the uploads, the kernels and the downloads
    const bool tracing = c->trace || trace_env();
    const auto t_wall0 = std::chrono::steady_clock::now();
    nvtxRangePushA(P.name);
    struct NvtxPop { ~NvtxPop() { nvtxRangePop(); } } nvtx_pop;
    if (tracing && !c->ev_t[0]) for (int i = 0; i < 6; i++) BGSB_CUDA(cudaEventCreate(&c->ev_t[i]));
    auto mark = [&](int i, cudaStream_t st) { if (tracing) cudaEventRecord(c->ev_t[i], st); };
    if (nchunks == 1) {
        mark(0, c->stream);
        if (fmt != BGSB_INPUT_BGR) BGSB_CUDA(upload_yuv(fmt, c->d_yuv, bgr, stride, w, h, 0, h, c->nstreams, c->stream));
        else BGSB_CUDA(copy_rows(d_up, (size_t)w * 3, bgr, stride, (size_t)w * 3, rows, cudaMemcpyHostToDevice, c->stream));
        mark(1, c->stream); mark(2, c->stream);
        if (fmt != BGSB_INPUT_BGR) {
            rc = convert_yuv(fmt, c->d_yuv, w, h, 0, h, c->nstreams, d_up, c->stream);
            if (rc) return rc;
        }
        if (blur) {            // also on warm-up frames that launch no plugin kernel: the ring slot becomes history
            rc = blur_frames(c->d_prep, w, h, 0, h, c->nstreams, d_in, c->stream);
            if (rc) return rc;
        }
        if (out_fg || P.warmup_launch) {
            rc = launch_range(c, d_in, 1, c->d_fg, want_bg ? c->d_bg : nullptr, 0, own_hist, c->stream, 0, c->npx);
            if (rc) return rc;
        }
        mark(3, c->stream); mark(4, c->stream);
        if (out_fg) {
            BGSB_CUDA(copy_rows(fg, fg_stride, c->d_fg, (size_t)w, (size_t)w, rows, cudaMemcpyDeviceToHost, c->stream));
            if (want_bg)
                BGSB_CUDA(copy_rows(bg, bg_stride, c->d_bg, bgw, bgw, rows, cudaMemcpyDeviceToHost, c->stream));
        }
        mark(5, c->stream);
        BGSB_CUDA(cudaStreamSynchronize(c->stream));
    } else {
        // band i arrives (upload, then the YUV conversion on the kernel stream), then band i's kernels run; with the blur
        // they run one band later, because band i's blur reads up to 3 rows of band i + 1 (bands are >= 32 rows)
        const int lag = blur ? 1 : 0;
        for (int it = 0; it < nchunks + lag; it++) {
            if (it < nchunks) {
                const int r0 = it * band, nr = std::min(band, h - r0);
                const size_t p0 = (size_t)r0 * w;
                if (it == 0) mark(0, c->s_h2d);
                if (fmt != BGSB_INPUT_BGR) BGSB_CUDA(upload_yuv(fmt, c->d_yuv, bgr, stride, w, h, r0, nr, 1, c->s_h2d));
                else BGSB_CUDA(copy_rows(d_up + p0 * 3, (size_t)w * 3, bgr + (size_t)r0 * stride, stride, (size_t)w * 3, nr,
                                         cudaMemcpyHostToDevice, c->s_h2d));
                BGSB_CUDA(cudaEventRecord(c->ev_up[it], c->s_h2d));
                if (it == nchunks - 1) mark(1, c->s_h2d);
                BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_up[it], 0));
                if (it == 0) mark(2, c->stream);
                if (fmt != BGSB_INPUT_BGR) {       // bands are multiples of 32 rows: whole chroma rows
                    rc = convert_yuv(fmt, c->d_yuv, w, h, r0, nr, 1, d_up, c->stream);
                    if (rc) return rc;
                }
            }
            const int i = it - lag;
            if (i < 0) continue;
            const int r0 = i * band, nr = std::min(band, h - r0);
            const size_t p0 = (size_t)r0 * w;
            if (blur) {
                rc = blur_frames(c->d_prep, w, h, r0, nr, 1, d_in, c->stream);
                if (rc) return rc;
            }
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
            fprintf(stderr, "%s\ttime(sec):%.6f\tupload %.6f kernels %.6f download %.6f (%d band%s, stages overlap)\n", P.name,
                    T.wall_ms * 1e-3, up * 1e-3, kn * 1e-3, dn * 1e-3, nchunks, nchunks > 1 ? "s" : "");
    }
    advance(c, 1, own_hist);
    if (P.ring_history) remember_input(c, d_in);
    if (fg_valid) *fg_valid = out_fg;
    if (bg_valid) *bg_valid = want_bg;
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
    int rc = check_host_frame(c, bgr, w, h, stride, fg, fg_stride, bg, bg_stride);
    if (rc) return rc;
    BGSB_CUDA(cudaSetDevice(c->device));
    if (c->w != w || c->h != h) {                                  // geometry change: nothing may be in flight
        rc = drain(c);
        if (rc) return rc;
    }
    rc = host_setup(c, w, h);
    if (rc) return rc;
    const size_t S = (size_t)c->nstreams;
    {
        cudaError_t e = cudaSuccess;
        if (!c->d_fg2) e = cudaMalloc(&c->d_fg2, S * c->npx);
        if (e == cudaSuccess && !c->d_bg2 && c->d_bg) e = cudaMalloc(&c->d_bg2, S * c->npx * 3);
        if (e != cudaSuccess) { drain(c); return staging_fail(c, e); }
    }
    const PluginInfo &P = *c->pi;
    const size_t rows = (size_t)h * c->nstreams;
    const size_t bgw = (size_t)w * P.bg_channels;
    uint8_t *d_in = c->d_ring[c->ring_pos];
    const bool out_fg = mask_due(c), want_bg = bg_due(c, bg);
    const bool own_hist = !P.ring_history;
    const int slot = (int)(c->seq & 1);
    uint8_t *o_fg = slot ? c->d_fg2 : c->d_fg, *o_bg = slot ? c->d_bg2 : c->d_bg;
    const int fmt = c->input_format;
    if (fmt != BGSB_INPUT_BGR && (rc = ensure_yuv_staging(c))) { drain(c); return rc; }
    const bool blur = c->gaussian_blur != 0;
    if (blur && (rc = ensure_prep_staging(c))) { drain(c); return rc; }
    uint8_t *const d_up = blur ? c->d_prep : d_in;

    // the input buffer (ring slot, or the YUV / blur staging) was last read by the previous frame's kernels
    if (c->seq > 0) BGSB_CUDA(cudaStreamWaitEvent(c->s_h2d, c->ev_k[slot ^ 1], 0));
    if (fmt != BGSB_INPUT_BGR) BGSB_CUDA(upload_yuv(fmt, c->d_yuv, bgr, stride, w, h, 0, h, c->nstreams, c->s_h2d));
    else BGSB_CUDA(copy_rows(d_up, (size_t)w * 3, bgr, stride, (size_t)w * 3, rows, cudaMemcpyHostToDevice, c->s_h2d));
    BGSB_CUDA(cudaEventRecord(c->ev_up[slot], c->s_h2d));
    BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_up[slot], 0));
    if (fmt != BGSB_INPUT_BGR) {
        rc = convert_yuv(fmt, c->d_yuv, w, h, 0, h, c->nstreams, d_up, c->stream);
        if (rc) return rc;
    }
    if (blur) {
        rc = blur_frames(c->d_prep, w, h, 0, h, c->nstreams, d_in, c->stream);
        if (rc) return rc;
    }
    if (out_fg || P.warmup_launch) {
        BGSB_CUDA(cudaStreamWaitEvent(c->stream, c->ev_dn[slot], 0));       // output slot free (no-op until recorded)
        rc = launch_range(c, d_in, 1, o_fg, want_bg ? o_bg : nullptr, 0, own_hist, c->stream, 0, c->npx);
        if (rc) return rc;
    }
    BGSB_CUDA(cudaEventRecord(c->ev_k[slot], c->stream));
    if (out_fg) {
        BGSB_CUDA(cudaStreamWaitEvent(c->s_d2h, c->ev_k[slot], 0));
        BGSB_CUDA(copy_rows(fg, fg_stride, o_fg, (size_t)w, (size_t)w, rows, cudaMemcpyDeviceToHost, c->s_d2h));
        if (want_bg) BGSB_CUDA(copy_rows(bg, bg_stride, o_bg, bgw, bgw, rows, cudaMemcpyDeviceToHost, c->s_d2h));
        BGSB_CUDA(cudaEventRecord(c->ev_dn[slot], c->s_d2h));
    }
    advance(c, 1, own_hist);
    if (P.ring_history) remember_input(c, d_in);
    c->seq += 1;
    c->inflight = true;
    if (fg_valid) *fg_valid = out_fg;
    if (bg_valid) *bg_valid = want_bg;
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
    for (int k = 0; k < n; k++) BGSB_REQUIRE(ctxs[k], "null ctx");
    bgsb_ctx *c0 = ctxs[0];
    const int fmt = c0->input_format;      // YUV: each band is uploaded once and converted once into the shared frame
    if (fmt != BGSB_INPUT_BGR) {
        int rc = check_yuv_frame(fmt, w, h, stride);
        if (rc) return rc;
    }
    BGSB_REQUIRE(stride >= (size_t)w * (fmt == BGSB_INPUT_BGR ? 3 : 1), "stride smaller than a row");
    for (int k = 0; k < n; k++)
        BGSB_REQUIRE(ctxs[k]->input_format == fmt, "fan-out contexts must share one \"inputFormat\"");
    const bool blur = c0->gaussian_blur != 0;  // blur: each band lands in c0's d_prep and is blurred once into the shared frame
    for (int k = 0; k < n; k++)
        BGSB_REQUIRE((ctxs[k]->gaussian_blur != 0) == blur, "fan-out contexts must share one \"gaussianBlur\"");
    for (int k = 0; k < n; k++) { if (int drc = drain(ctxs[k])) return drc; }
    for (int k = 0; k < n; k++) {
        BGSB_REQUIRE(ctxs[k] && fg[k], "null context or mask buffer");
        BGSB_REQUIRE(ctxs[k]->device == c0->device && ctxs[k]->nstreams == 1, "fan-out takes single-stream contexts of one device");
        BGSB_REQUIRE(fg_stride[k] >= (size_t)w, "fg stride smaller than a row");
        BGSB_REQUIRE(!(bg && bg[k]) || (bg_stride && bg_stride[k] >= (size_t)w * ctxs[k]->pi->bg_channels),
                     "bg stride smaller than a row");
        for (int j = 0; j < k; j++) BGSB_REQUIRE(ctxs[j] != ctxs[k], "the same context twice");
    }
    BGSB_CUDA(cudaSetDevice(c0->device));
    for (int k = 0; k < n; k++) {
        int rc = host_setup(ctxs[k], w, h);
        if (rc) return rc;
    }
    if (fmt != BGSB_INPUT_BGR) {
        int rc = ensure_yuv_staging(c0);
        if (rc) return rc;
    }
    if (blur) {
        int rc = ensure_prep_staging(c0);
        if (rc) return rc;
    }
    const size_t fbytes = (size_t)w * h * 3;
    if (c0->d_fan_bytes < fbytes) {
        cudaFree(c0->d_fan); c0->d_fan = nullptr; c0->d_fan_bytes = 0;
        BGSB_CUDA(cudaMalloc(&c0->d_fan, fbytes));
        c0->d_fan_bytes = fbytes;
    }
    // row bands as in bgsb_process, as many as the first context's "hostBands" (2 unless set): the upload of band i+1
    // overlaps the n kernels on band i (each on its own context's stream) and the downloads of band i-1
    const Bands B = plan_bands(w, h, c0->host_bands);
    const int nchunks = B.n, band = B.rows;
    bool fgv[16], bgv[16];
    for (int k = 0; k < n; k++) {
        fgv[k] = mask_due(ctxs[k]);
        bgv[k] = bg_due(ctxs[k], bg ? bg[k] : nullptr);
    }
    uint8_t *const d_up = blur ? c0->d_prep : c0->d_fan;
    const int lag = blur ? 1 : 0;        // band i's blur reads up to 3 rows of band i + 1, as in bgsb_process
    for (int it = 0; it < nchunks + lag; it++) {
        if (it < nchunks) {
            const int r0 = it * band, nr = std::min(band, h - r0);
            const size_t p0 = (size_t)r0 * w;
            if (fmt != BGSB_INPUT_BGR) {
                BGSB_CUDA(upload_yuv(fmt, c0->d_yuv, bgr, stride, w, h, r0, nr, 1, c0->s_h2d));
                int rc = convert_yuv(fmt, c0->d_yuv, w, h, r0, nr, 1, d_up, c0->s_h2d);
                if (rc) return rc;
            } else {
                BGSB_CUDA(copy_rows(d_up + p0 * 3, (size_t)w * 3, bgr + (size_t)r0 * stride, stride, (size_t)w * 3, nr,
                                    cudaMemcpyHostToDevice, c0->s_h2d));
            }
        }
        const int i = it - lag;
        if (i < 0) continue;
        const int r0 = i * band, nr = std::min(band, h - r0);
        const size_t p0 = (size_t)r0 * w;
        if (blur) {
            int rc = blur_frames(c0->d_prep, w, h, r0, nr, 1, c0->d_fan, c0->s_h2d);
            if (rc) return rc;
        }
        BGSB_CUDA(cudaEventRecord(c0->ev_up[i], c0->s_h2d));
        for (int k = 0; k < n; k++) {
            bgsb_ctx *c = ctxs[k];
            BGSB_CUDA(cudaStreamWaitEvent(c->stream, c0->ev_up[i], 0));
            // a plugin whose mask needs neighbouring pixels (3x3 median) runs once, on the whole frame, after the
            // last band has arrived
            const bool whole = c->pi->stencil;
            if (whole && i != nchunks - 1) continue;
            const size_t q0 = whole ? 0 : p0;
            const int qr0 = whole ? 0 : r0, qnr = whole ? h : nr;
            const size_t bgw = (size_t)w * c->pi->bg_channels;
            // the frame buffer is shared, so every plugin keeps its own history (FD / WMV copy the frame); d_bg is null
            // for a plugin that writes no background
            int rc = launch_range(c, c0->d_fan, 1, c->d_fg, c->d_bg, 0, true, c->stream, q0, qnr * w);
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
    BGSB_REQUIRE(w > 0 && h > 0, "empty frame");
    // a mode count above K would make the kernels walk past the pixel's K modes: refused before anything changes
    for (size_t i = 0, n = (size_t)w * h; i < n; i++)
        BGSB_REQUIRE(nmodes[i] <= MOG2_K, "nmodes above 5");
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
    cudaStream_t su = nullptr, sd = nullptr;
    cudaError_t e = cudaHostAlloc(&h_up, bytes_up, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaHostAlloc(&h_dn, bytes_down, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaMalloc(&d_up, bytes_up);
    if (e == cudaSuccess) e = cudaMalloc(&d_dn, bytes_down);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&su, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&sd, cudaStreamNonBlocking);
    if (e == cudaSuccess) { memset(h_up, 1, bytes_up); memset(h_dn, 0, bytes_down); }
    auto issue = [&](bool up, bool down) {
        if (up && e == cudaSuccess) e = cudaMemcpyAsync(d_up, h_up, bytes_up, cudaMemcpyHostToDevice, su);
        if (down && e == cudaSuccess) e = cudaMemcpyAsync(h_dn, d_dn, bytes_down, cudaMemcpyDeviceToHost, sd);
    };
    auto sync_all = [&]() {
        if (e == cudaSuccess) e = cudaStreamSynchronize(su);
        if (e == cudaSuccess) e = cudaStreamSynchronize(sd);
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
    if (su) cudaStreamDestroy(su);
    if (sd) cudaStreamDestroy(sd);
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
