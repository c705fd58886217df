/*
 * bgsb200 -- B200-native (sm_100a) foreground-extraction hot path, C ABI.
 *
 * This is the drop-in boundary below the reference's C++ plugin interfaces.  Every entry
 * point names the reference interface it replaces (paths relative to the reference tree):
 *
 *   IBGS::process(const cv::Mat&, cv::Mat&, cv::Mat&)            package_bgs/IBGS.h:24
 *     FrameDifferenceBGS::process                                 package_bgs/FrameDifferenceBGS.cpp:29-61
 *     AdaptiveBackgroundLearning::process                         package_bgs/AdaptiveBackgroundLearning.cpp:30-83
 *     StaticFrameDifferenceBGS::process  (sibling, 8f N3)          package_bgs/StaticFrameDifferenceBGS.cpp:29-57
 *     WeightedMovingMeanBGS::process     (sibling, 8f N3)          package_bgs/WeightedMovingMeanBGS.cpp:30-103
 *     WeightedMovingVarianceBGS::process                          package_bgs/WeightedMovingVarianceBGS.cpp:30-117
 *     MixtureOfGaussianV2BGS::process                             package_bgs/MixtureOfGaussianV2BGS.cpp:29-74
 *   USTC_BGS::Process / GetMask / Release (CvFGDetector)          ustc_src/ustc_bgs.cpp:75-113
 *   cv::erode / cv::dilate on the foreground mask                 package_bgs/jmo/CMultiLayerBGS.cpp:1614-1615 (and SURVEY 8a row aM)
 *   CvBlobDetector::DetectNewBlob (cvCreateBlobDetectorCC)        ustc_src/trackingMain.cpp:56,626
 *
 * Plain C types only; `int` status (0 = BGSB_OK); the caller owns every I/O buffer, the
 * library owns all model state; one context = one group of independent camera streams on
 * one GPU.  A context is not thread-safe; distinct contexts are.  There is NO CPU fallback:
 * every call that computes runs CUDA kernels and fails with BGSB_ERR_CUDA without a GPU.
 *
 * The header-only C++ adapters in tracking_b200/adapters/ re-declare the reference's
 * classes on top of this ABI; INTEGRATION.md shows the binding a maintainer adds.
 */
#ifndef BGSB200_H
#define BGSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define BGSB_API
#else
#define BGSB_API __attribute__((visibility("default")))
#endif

/* status codes */
enum {
    BGSB_OK = 0,
    BGSB_ERR_ARG = 1,      /* bad argument (null pointer, bad size, unknown key/algo) */
    BGSB_ERR_CUDA = 2,     /* CUDA runtime error, text in bgsb_last_error() */
    BGSB_ERR_STATE = 3,    /* call not valid in the context's current state */
    BGSB_ERR_CAPACITY = 4  /* a caller-provided table was too small */
};

/* algorithm ids == the integer ids of the USTC_BGS factory (ustc_src/ustc_bgs.cpp:8-14) */
enum {
    BGSB_ALGO_FRAME_DIFFERENCE = 0,           /* ustc_bgs.cpp:8  */
    BGSB_ALGO_STATIC_FRAME_DIFFERENCE = 1,    /* ustc_bgs.cpp:9   sibling plugin (SURVEY 8f N3) */
    BGSB_ALGO_WEIGHTED_MOVING_MEAN = 2,       /* ustc_bgs.cpp:10  sibling plugin (SURVEY 8f N3) */
    BGSB_ALGO_WEIGHTED_MOVING_VARIANCE = 3,   /* ustc_bgs.cpp:11 */
    BGSB_ALGO_MOG2 = 5,                       /* ustc_bgs.cpp:13 */
    BGSB_ALGO_ADAPTIVE_BG_LEARNING = 6,       /* ustc_bgs.cpp:14 */
    BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING = 7, /* ustc_bgs.cpp:15  sibling plugin (SURVEY 8f N3); gray 1-channel bg image */
    BGSB_ALGO_DP_ADAPTIVE_MEDIAN = 9,             /* ustc_bgs.cpp:19  sibling plugin (DP package); never writes img_bgmodel */
    BGSB_ALGO_DP_ZIVKOVIC_AGMM = 11,              /* ustc_bgs.cpp:21  sibling plugin (SURVEY 8f N3); never writes img_bgmodel */
    BGSB_ALGO_DP_MEAN = 12,                       /* ustc_bgs.cpp:22  sibling plugin (DP package); never writes img_bgmodel */
    BGSB_ALGO_DP_WREN_GA = 13,                    /* ustc_bgs.cpp:23  sibling plugin (DP package); never writes img_bgmodel */
    BGSB_ALGO_DP_PRATI_MEDIOD = 14,               /* ustc_bgs.cpp:24  sibling plugin (DP package); never writes img_bgmodel */
    BGSB_ALGO_SIGMA_DELTA = 35                    /* ustc_bgs.cpp:62  sibling plugin (BL package); first frame: no outputs */
};

/* Values of the "inputFormat" parameter (bgsb_set_param): the layout of the frames a context's calls take.
 *   BGSB_INPUT_BGR  : interleaved BGR, 3 bytes per pixel (default).
 *   BGSB_INPUT_NV12 : YUV 4:2:0 as NVDEC, V4L2 and most camera SDKs produce it: h rows of w Y bytes, then h/2 rows of w
 *                     bytes of interleaved U,V; on host paths both kinds of row sit `stride` bytes apart.
 *   BGSB_INPUT_I420 : YUV 4:2:0 planar (ffmpeg's AV_PIX_FMT_YUV420P): the Y plane (w x h), the U plane (w/2 x h/2), the V
 *                     plane, densely packed; on host paths `stride` must equal w.
 * Both are one 8-bit image of 3h/2 rows of w bytes, the cv::Mat that cv::cvtColor(COLOR_YUV2BGR_NV12 / _I420) reads; w
 * and h must be even.  Device buffers are dense: [nstreams][3h/2][w], and [nstreams][T][3h/2][w] for batches.  The
 * library converts each frame on the device to exactly the BGR image cv::cvtColor gives (BT.601, limited range,
 * 20-bit fixed point) and runs the plugin on it, so every result equals that of the BGR path fed cv::cvtColor's output. */
enum { BGSB_INPUT_BGR = 0, BGSB_INPUT_NV12 = 1, BGSB_INPUT_I420 = 2 };

typedef struct bgsb_ctx bgsb_ctx;

/* ---------------------------------------------------------------------------------------
 * Library / device
 * ------------------------------------------------------------------------------------- */
BGSB_API const char *bgsb_last_error(void);          /* thread-local text of the last failure */
BGSB_API const char *bgsb_version(void);
BGSB_API int bgsb_device_count(int *count);
/* Page-locked host memory for frame staging (the capture side of the boundary, SURVEY 8f N1): uploads from
 * pinned buffers are true DMA.  write_combined != 0 allocates write-combined memory (fast for the CPU to
 * fill sequentially and for the GPU to read, slow for the CPU to read back: use it for INPUT frames only). */
BGSB_API int bgsb_host_alloc(void **ptr, size_t bytes, int write_combined);
BGSB_API void bgsb_host_free(void *ptr);
/* Diagnostic: what the PCIe link of `device` sustains from this process -- seconds per iteration for a page-locked
 * upload of bytes_up alone, a download of bytes_down alone, and both at once on two streams (no kernels).  The host-
 * buffer entry points (bgsb_process, bgsb_submit, bgsb_pool_*) cannot be faster than max(up, down) per frame. */
BGSB_API int bgsb_copy_probe(int device, size_t bytes_up, size_t bytes_down, int iters, double *sec_up, double *sec_down,
                             double *sec_both);
/* Number of kernels this library has launched in the calling process (bench.py gpu_launches). */
BGSB_API uint64_t bgsb_kernel_launch_count(void);

/* ---------------------------------------------------------------------------------------
 * Background-subtraction contexts  (replaces `new <Plugin>` / `delete`,
 * FrameProcessor.cpp:40-59,459-478; ustc_src/ustc_bgs.cpp:8-14,75-77)
 * ------------------------------------------------------------------------------------- */
/* One camera stream. */
BGSB_API int bgsb_create(bgsb_ctx **out, int algo, int device);
/* `nstreams` independent camera streams of identical geometry that are advanced together
 * by one launch per frame (stream group; SURVEY 8e).  Stream s of every *_dev buffer below
 * sits at base + s * (per-stream bytes). */
BGSB_API int bgsb_create_group(bgsb_ctx **out, int algo, int device, int nstreams);
BGSB_API void bgsb_destroy(bgsb_ctx *ctx);
/* Drop all model state (next frame is frame 0 again). */
BGSB_API int bgsb_reset(bgsb_ctx *ctx);

/* Parameters carry the reference's XML key names (saveConfig/loadConfig of each plugin):
 *   all      : "enableThreshold" (1), "threshold" (15)
 *   MOG2     : "alpha" (0.05)             MixtureOfGaussianV2BGS.cpp:92-95
 *              (as cv::BackgroundSubtractorMOG2::apply: alpha >= 1 re-initialises the model before every frame, which then
 *              learns at 1/min(2, history); after it, alpha < 0 counts its automatic rate from that frame again)
 *   ABL      : "alpha" (0.05), "limit" (-1; only -1 updates the model, .cpp:52)
 *   DPZivkovicAGMM : "threshold" (25.0), "alpha" (0.001), "gaussians" (3, at most 5)   DPZivkovicAGMMBGS.cpp:86-100
 *              (latched at the first frame like the reference's params hand-over, .cpp:58-65: a later change takes
 *              effect after bgsb_reset)
 *   ASBL     : "learningFrames" (90), "alphaLearn" (0.05), "alphaDetection" (0.05), "threshold" (25)
 *              AdaptiveSelectiveBackgroundLearning.cpp:108-126 (the defaults its loadConfig applies)
 *   WMV, WMM : "enableWeight" (1)         WeightedMovingVarianceBGS.cpp:155-158, WeightedMovingMeanBGS.cpp
 * plus the cv::BackgroundSubtractorMOG2 properties of the default-constructed member
 * (MixtureOfGaussianV2BGS.h:30): "history" 500, "nmixtures" 5 (fixed), "varThreshold" 16,
 * "varThresholdGen" 9, "backgroundRatio" 0.9, "varInit" 15, "varMin" 4, "varMax" 75,
 * "complexityReductionThreshold" 0.05, "detectShadows" 1, "shadowValue" 127,
 * "shadowThreshold" 0.5 (varMin / varMax given in the wrong order are swapped, as OpenCV does); and "grayVariant": 0 = OpenCV 4.x BGR2GRAY constants, 1 = 2.4.x;
 * "kernelVariant" (MOG2): 0 = production kernels, 1 = straight restatement kernel (identical results, kept for
 * A/B measurements; any other value is refused);
 * "ablTable" (AdaptiveBackgroundLearning): 1 = lookup-table kernels (default), 2 = only the per-thread table kernel,
 * 3 = as 1, with the bulk-copy kernel whenever the geometry allows (by default only for groups of ~3.6 Mpx and more),
 * 0 = arithmetic kernel -- identical results;
 * "ablBlend" (AdaptiveBackgroundLearning): 0 = cv::addWeighted as OpenCV 4.x computes it (double precision; pinned
 * against cv2 4.13, default), 1 = as OpenCV 2.4 does (fp32 arithmetic, scalars cast to float; SURVEY Appendix B --
 * "parity unpinned": no OpenCV 2.4 in the build image), table kernels only;
 * "hostBands" (1..8; default: 3 when the background image is returned too, else 2): row bands of the upload / kernel /
 * download pipeline inside bgsb_process;
 * "trace" (default 0): per-stage timing of bgsb_process, see bgsb_trace_last;
 * "quietGroups" (WeightedMovingVariance, default 1): with the threshold on, a 16-pixel group whose bytes moved by at most
 * R over the three frames gets its all-zero mask without the arithmetic; R is derived from the threshold by running all
 * 2^24 byte triples through the kernel's own routine once per weight set (identical results; 0 = always compute);
 * AdaptiveBackgroundLearning's table kernel uses the same switch: 16 model bytes that all lie within the table's quiet
 * radius of the input (largest D with blend(x, y) == y for |x - y| <= D, read off the finished table on the device:
 * 9 at alpha 0.05) are kept without the 16 lookups;
 * "retainInput" (default 0; FrameDifference, WeightedMovingVariance, WeightedMovingMean on the *_dev entry points):
 * 1 = the caller promises that the device frame given to a call stays valid and unmodified until the next call (FD)
 * / the next two calls (WMV, WMM) have completed, so the previous-frame history is read from those buffers and never
 * copied (the reference's img_input_prev members, FrameDifferenceBGS.cpp:58, WeightedMovingVarianceBGS.cpp:113-114):
 * FD moves 7 B/px instead of 10, WMV 10 instead of 16.  Single frames, or batches on a single-stream context;
 * "inputFormat" (default BGSB_INPUT_BGR): BGSB_INPUT_NV12 / BGSB_INPUT_I420 make every entry point (bgsb_process,
 * bgsb_submit, bgsb_process_fanout, bgsb_process_dev, bgsb_process_batch_dev, the pipeline and the pool) take YUV 4:2:0
 * frames (see the enum above).  The host paths upload 1.5 B/px instead of 3 and convert on the device into the buffer
 * the BGR upload would fill; the device paths convert into a library-owned scratch on the caller's stream first.  The
 * model and the history are kept as BGR, so the format may change between calls.  BGSB_ERR_ARG for an odd w or h, an
 * I420 host frame with stride != w, and together with "retainInput" (the converted frames are the library's, so the
 * caller's buffers cannot serve as the history).  Fan-out contexts must share one format;
 * "gaussianBlur" (0 or 1, default 0): the reference PreProcessor's gaussianBlur switch (FrameProcessor.cpp:173-174).  1 =
 * every frame is blurred on the device, exactly as cv::GaussianBlur(img, Size(7, 7), 1.5) does on 8-bit BGR (OpenCV 4.x,
 * BORDER_REFLECT_101), before the plugin sees it: on every entry point, after the YUV conversion with a YUV
 * "inputFormat", and on warm-up frames too, so the history FrameDifference / WeightedMovingVariance / WeightedMovingMean
 * keep is the blurred frame.  A change takes effect from the next frame.  The host paths upload into a staging buffer
 * and blur into the buffer the upload would fill; the device paths blur into a library-owned scratch on the caller's
 * stream.  BGSB_ERR_ARG for any other value, and together with "retainInput" in either order (the history is the
 * blurred frame, so the caller's buffers cannot serve as it).  Fan-out contexts must share one value.  A C++ caller that
 * keeps FrameProcessor's PreProcessor with only gaussianBlur enabled sets this key on each GPU plugin and hands them
 * img_input instead of img_prep (INTEGRATION.md 4b). */
BGSB_API int bgsb_set_param(bgsb_ctx *ctx, const char *key, double value);
BGSB_API int bgsb_get_param(bgsb_ctx *ctx, const char *key, double *value);

/* IBGS::process with HOST buffers, synchronous (outputs complete on return).
 *   bgr        : h rows of w BGR pixels, `stride` bytes between rows (cv::Mat::step)
 *   fg         : h x w 8UC1, fg_stride bytes between rows
 *   bg         : h x w 8UC3 (8UC1 for BGSB_ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING, whose model is gray), may be NULL
 *   *fg_valid  : 0 reproduces "output left untouched" (FD frame 0, WMV frames 0-1:
 *                FrameDifferenceBGS.cpp:39-43, WeightedMovingVarianceBGS.cpp:40-51)
 *   *bg_valid  : 0 for FD / WMV, which never write img_bgmodel (StaticFD / WMM / ABL / MOG2 do)
 * For a stream group the buffers hold nstreams images back to back (stride * h bytes each). */
BGSB_API int bgsb_process(bgsb_ctx *ctx, const uint8_t *bgr, int w, int h, size_t stride,
                          uint8_t *fg, size_t fg_stride, uint8_t *bg, size_t bg_stride,
                          int *fg_valid, int *bg_valid);

/* Pipelined ingest for the capture loop (VideoCapture.cpp:151-239 reads a frame and calls FrameProcessor::process;
 * ustc_src/trackingMain.cpp:161-166 does the same with cvQueryFrame + USTC_BGS::Process): bgsb_process, queued.
 * bgsb_submit returns once the frame's upload, kernel and downloads are enqueued; the upload of the next frame then
 * overlaps the download of this one (a synchronous call cannot use both PCIe directions at once).  The model
 * advances in submission order: results are those of the same sequence of bgsb_process calls.  Arguments as in
 * bgsb_process; bgr / fg / bg must stay valid and untouched until bgsb_wait returns and should be page-locked
 * (bgsb_host_alloc).  *fg_valid / *bg_valid are known at submission.  Any number of frames may be queued; every other
 * entry point taking this context waits for them first.
 * bgsb_wait: all submitted frames' outputs are in their host buffers. */
BGSB_API int bgsb_submit(bgsb_ctx *ctx, const uint8_t *bgr, int w, int h, size_t stride,
                         uint8_t *fg, size_t fg_stride, uint8_t *bg, size_t bg_stride,
                         int *fg_valid, int *bg_valid);
BGSB_API int bgsb_wait(bgsb_ctx *ctx);

/* FrameProcessor::process (FrameProcessor.cpp:169-215) runs every enabled plugin back to back on the same
 * prepared frame.  Fan-out does that with ONE upload: the frame goes to the device once (in row bands), the n
 * contexts' kernels run on it concurrently, and each plugin's outputs come back as in bgsb_process.
 * Results and per-context state are identical to calling bgsb_process on each context.
 *   ctxs[n]      : single-stream contexts on one device (any mix of algorithms), n <= 16
 *   fg[n], bg[n] : per-context output buffers (bg or bg[k] may be NULL), with their row strides
 *   fg_valid[n], bg_valid[n] : as in bgsb_process, may be NULL */
BGSB_API int bgsb_process_fanout(bgsb_ctx *const *ctxs, int n, const uint8_t *bgr, int w, int h, size_t stride,
                                 uint8_t *const *fg, const size_t *fg_stride,
                                 uint8_t *const *bg, const size_t *bg_stride,
                                 int *fg_valid, int *bg_valid);

/* Same, DEVICE buffers, dense rows (stride == 3*w / w), asynchronous on `stream`
 * (a cudaStream_t; NULL = legacy default stream).  d_bg may be NULL. */
BGSB_API int bgsb_process_dev(bgsb_ctx *ctx, const uint8_t *d_bgr, int w, int h,
                              uint8_t *d_fg, uint8_t *d_bg, int *fg_valid, int *bg_valid,
                              void *stream);

/* Temporal batch: T consecutive frames per stream in ONE launch; the per-pixel model
 * state stays in registers across the T frames and is read and written once.
 *   d_frames : [nstreams][T][h][w][3]     d_fg : [nstreams][T][h][w]
 *   d_bg     : [nstreams][T][h][w][3], or NULL
 *   bg_last_only != 0 : d_bg is [nstreams][h][w][3] and receives only frame T-1's model
 *   *first_fg_valid : index of the first frame of the batch whose mask was written
 *                     (0 normally; 1 / 2 while FD / WMV warm up; T if none). */
BGSB_API int bgsb_process_batch_dev(bgsb_ctx *ctx, const uint8_t *d_frames, int T, int w, int h,
                                    uint8_t *d_fg, uint8_t *d_bg, int bg_last_only,
                                    int *first_fg_valid, int *bg_valid, void *stream);

/* Tracing (FrameProcessor::tic / toc, FrameProcessor.cpp:484-494, which times one plugin's process() call on the host and
 * keeps working unchanged around the drop-in): with the context parameter "trace" = 1, or BGSB_TRACE=1 in the
 * environment, every bgsb_process call is also timed per stage on the device (CUDA events around the uploads, the
 * kernels and the downloads; with row bands the stages overlap, so they need not add up to the wall time).
 * BGSB_TRACE=1 prints toc's line "<Plugin>\ttime(sec):<s>" plus the stage split on stderr.  Every entry point that
 * enqueues work is wrapped in an NVTX range named after the plugin (visible in Nsight Systems). */
typedef struct bgsb_trace {
    int64_t frame;          /* index of the traced frame */
    double wall_ms;         /* host wall time of the call */
    double upload_ms, kernel_ms, download_ms;
    int bands;              /* row bands of the call's upload / kernel / download pipeline */
} bgsb_trace;
BGSB_API int bgsb_trace_last(bgsb_ctx *ctx, bgsb_trace *out);

/* Number of frames this context has consumed since create/reset. */
BGSB_API int bgsb_frame_count(bgsb_ctx *ctx, int64_t *nframes);
/* Bytes of HBM model state held per stream (101 B/px for MOG2). */
BGSB_API int bgsb_state_bytes(bgsb_ctx *ctx, size_t *bytes);
/* Raw MOG2 state export/import (SURVEY 8f N4): K planes each of weight, variance,
 * mean B, G, R as fp32 [25][npx] followed by nmodes u8 [npx]; host buffers.
 * Import refuses a mode count above 5 (BGSB_ERR_ARG) and then leaves the context as it was. */
BGSB_API int bgsb_mog2_export_state(bgsb_ctx *ctx, int stream_index, float *planes, uint8_t *nmodes);
BGSB_API int bgsb_mog2_import_state(bgsb_ctx *ctx, int stream_index, int w, int h, int64_t nframes,
                                    const float *planes, const uint8_t *nmodes);

/* ---------------------------------------------------------------------------------------
 * Mask morphology (cv::erode / cv::dilate, default 3x3 rect element, SURVEY A.5)
 *   ops[2*i] = BGSB_MORPH_ERODE | BGSB_MORPH_DILATE, ops[2*i+1] = iterations (>= 0)
 *   masks are {0,255} bytes; any non-zero input byte counts as set.
 * ------------------------------------------------------------------------------------- */
enum { BGSB_MORPH_ERODE = 0, BGSB_MORPH_DILATE = 1 };
BGSB_API int bgsb_morph_dev(const uint8_t *d_mask, int w, int h, int nimages, const int *ops,
                            int nops, uint8_t *d_out, void *stream);
BGSB_API int bgsb_morph(const uint8_t *mask, int w, int h, size_t stride, const int *ops,
                        int nops, uint8_t *out, size_t out_stride);

/* ---------------------------------------------------------------------------------------
 * Connected components (steps 1-2 and the integer sums of step 4 of
 * CvBlobDetectorCC::DetectNewBlob, SURVEY A.6)
 * ------------------------------------------------------------------------------------- */
typedef struct bgsb_component {
    int32_t label;        /* canonical, 1-based: rank of the component's first raster pixel */
    int32_t first_index;  /* y*w + x of that pixel */
    int32_t x, y, w, h;   /* bounding rect (== CvContour::rect of the outer contour) */
    int32_t area;         /* pixel count */
    int32_t external;     /* 1 iff not enclosed in a hole of another component (RETR_EXTERNAL) */
} bgsb_component;

typedef struct bgsb_ccl bgsb_ccl;
BGSB_API int bgsb_ccl_create(bgsb_ccl **out, int device, int max_w, int max_h);
/* A labeller that can take up to max_images masks of one geometry per call (one launch sequence for
 * all camera streams of a group instead of one per stream). */
BGSB_API int bgsb_ccl_create_batch(bgsb_ccl **out, int device, int max_w, int max_h, int max_images);
BGSB_API void bgsb_ccl_destroy(bgsb_ccl *ccl);
/* "forceBackgroundPass" (default 0): label the background of every image for the RETR_EXTERNAL test even when
 * no bounding box lies inside another (A/B and tests; results are identical). */
BGSB_API int bgsb_ccl_set_param(bgsb_ccl *ccl, const char *key, double value);
/* foreground = mask > 128 (cvThreshold(pIB,pIB,128,255,BINARY)); 8-connected.
 * zero_border != 0 clears the outer 1-px frame first (OpenCV <= 3.1 cvFindContours).
 * d_labels (int32 [h][w], nullable) receives canonical labels, 0 = background.
 * Asynchronous on `stream`; the component table stays on the device until fetched. */
BGSB_API int bgsb_ccl_label_dev(bgsb_ccl *ccl, const uint8_t *d_mask, int w, int h, int zero_border,
                                int32_t *d_labels, void *stream);
/* nimages dense masks back to back ([nimages][h][w]); d_labels nullable, [nimages][h][w]. */
BGSB_API int bgsb_ccl_label_batch_dev(bgsb_ccl *ccl, const uint8_t *d_masks, int w, int h, int nimages,
                                      int zero_border, int32_t *d_labels, void *stream);
/* Synchronises `stream` and copies the component table (raster order) to the host. */
BGSB_API int bgsb_ccl_components(bgsb_ccl *ccl, bgsb_component *out, int capacity, int *n);
/* Same for image `image` of the last batch. */
BGSB_API int bgsb_ccl_components_of(bgsb_ccl *ccl, int image, bgsb_component *out, int capacity, int *n);
/* cvMoments(pFG[R], binary=0) for nrects rectangles of the mask last labelled:
 * out[6*i..] = m00 m10 m01 m20 m02 m11 (pixel-value weighted, ROI-relative, exact). */
BGSB_API int bgsb_ccl_rect_moments(bgsb_ccl *ccl, const int32_t *rects_xywh, int nrects, uint64_t *out);
/* Same for image `image` of the last batch. */
BGSB_API int bgsb_ccl_rect_moments_of(bgsb_ccl *ccl, int image, const int32_t *rects_xywh, int nrects, uint64_t *out);
/* Host-buffer convenience wrapper: label + fetch. */
BGSB_API int bgsb_ccl_label(bgsb_ccl *ccl, const uint8_t *mask, int w, int h, size_t stride,
                            int zero_border, int32_t *labels, bgsb_component *out, int capacity, int *n);

/* ---------------------------------------------------------------------------------------
 * CvBlobDetectorCC replacement (whole of SURVEY A.6; list logic on the host, CC + sums on GPU)
 * ------------------------------------------------------------------------------------- */
typedef struct bgsb_blob { float x, y, w, h; int32_t id; } bgsb_blob;   /* == CvBlob */
typedef struct bgsb_blobdetector bgsb_blobdetector;
BGSB_API int bgsb_blobdetector_create(bgsb_blobdetector **out, int device);
BGSB_API void bgsb_blobdetector_destroy(bgsb_blobdetector *bd);
/* keys: "HMin" 0.02, "WMin" 0.01, "MinDistToBorder" 1.1, "Clastering" 1, "Latency" 10,
 * "zeroBorder" 1 (OpenCV 2.4 cvFindContours behaviour) */
BGSB_API int bgsb_blobdetector_set_param(bgsb_blobdetector *bd, const char *key, double value);
/* DetectNewBlob(pImg, pFGMask, pNewBlobList, pOldBlobList) -> returns through *result the
 * reference's int result (1 = a new blob was appended to new_blobs).
 *   fg_mask host 8UC1; old_blobs = currently tracked blobs; new_blobs capacity >= 1.
 *   frame_blobs (nullable, capacity frame_cap) receives this frame's sorted top-10 list
 *   (m_pBlobLists[0]) for inspection / parity. */
BGSB_API int bgsb_blobdetector_detect(bgsb_blobdetector *bd, const uint8_t *fg_mask, int w, int h,
                                      size_t stride, const bgsb_blob *old_blobs, int n_old,
                                      bgsb_blob *new_blobs, int new_cap, int *n_new, int *result,
                                      bgsb_blob *frame_blobs, int frame_cap, int *n_frame);
/* Same with a device mask (dense), e.g. straight from bgsb_process_dev + bgsb_morph_dev. */
BGSB_API int bgsb_blobdetector_detect_dev(bgsb_blobdetector *bd, const uint8_t *d_fg_mask, int w, int h,
                                          const bgsb_blob *old_blobs, int n_old,
                                          bgsb_blob *new_blobs, int new_cap, int *n_new, int *result,
                                          bgsb_blob *frame_blobs, int frame_cap, int *n_frame,
                                          void *stream);

/* ---------------------------------------------------------------------------------------
 * The foreground pipeline, device-resident, for a group of camera streams: what the reference's main loop does per
 * frame (ustc_src/trackingMain.cpp:161-166 -> CvBlobTrackerAuto1::Process): USTC_BGS::Process = IBGS::process
 * (ustc_src/ustc_bgs.cpp:87-113), the mask clean-up (erode / dilate chain, SURVEY 8a row aM; default OPEN 3x3), and
 * steps 1-2 of CvBlobDetectorCC::DetectNewBlob (:626) -- BASELINE config 4.  The mask stays bit-packed between the
 * stages; one launch sequence serves all streams of the group.
 * ------------------------------------------------------------------------------------- */
typedef struct bgsb_pipeline bgsb_pipeline;
BGSB_API int bgsb_pipeline_create(bgsb_pipeline **out, int algo, int device, int nstreams);
BGSB_API void bgsb_pipeline_destroy(bgsb_pipeline *p);
/* The plugin context inside (owned by the pipeline): bgsb_set_param / bgsb_mog2_export_state ... on it. */
BGSB_API bgsb_ctx *bgsb_pipeline_bgs(bgsb_pipeline *p);
/* ops as in bgsb_morph_dev, at most 16 pairs; nops = 0: no clean-up stage. */
BGSB_API int bgsb_pipeline_set_morph(bgsb_pipeline *p, const int *ops, int nops);
/* "zeroBorder" (default 1, OpenCV 2.4 cvFindContours), "forceBackgroundPass", "chainCtas" (> 0: the labeller's
 * background pass as four plain launches of at most that many CTAs instead of one cooperative launch; default 0);
 * any other key goes to the plugin. */
BGSB_API int bgsb_pipeline_set_param(bgsb_pipeline *p, const char *key, double value);
/* One frame per stream: d_frames [nstreams][h][w][3].  Optional outputs (NULL = not wanted):
 *   d_mask   [nstreams][h][w]    the cleaned {0,255} mask (what CvFGDetector::GetMask hands to the tracker)
 *   d_bg     [nstreams][h][w][3] the plugin's background image
 *   d_labels [nstreams][h][w]    canonical labels of the 8-connected components (int32, 0 = background)
 * *valid = 0 while the plugin has no mask yet (FD frame 0, WMV frames 0-1): nothing was labelled.
 * With the plugin's "enableThreshold" 0 and a chain, the reference erodes / dilates the raw grey-level mask and
 * DetectNewBlob keeps what is > 128 afterwards: the pipeline labels exactly those pixels (it thresholds before the chain,
 * which commutes with erode / dilate), but it has no grey-level cleaned mask, so d_mask must be NULL (BGSB_ERR_ARG
 * otherwise) and bgsb_pipeline_rect_moments refuses that frame.  The stream pool inherits both.
 * Asynchronous.  The plugin kernel runs on `stream`; clean-up and labelling run on a stream of the pipeline behind
 * it, so that they overlap whatever the caller enqueues next on `stream` (normally the next frame's plugin kernel).
 * `stream` is made to wait for them only when d_mask or d_labels were given; otherwise the component tables (which
 * stay on the device until fetched) are ordered by the fetching calls below or by bgsb_pipeline_join_dev. */
BGSB_API int bgsb_pipeline_process_dev(bgsb_pipeline *p, const uint8_t *d_frames, int w, int h, uint8_t *d_mask,
                                       uint8_t *d_bg, int32_t *d_labels, int *valid, int *bg_valid, void *stream);
/* Make `stream` wait for everything the pipeline has enqueued so far (e.g. before an event that ends a timed region). */
BGSB_API int bgsb_pipeline_join_dev(bgsb_pipeline *p, void *stream);
/* Component table of stream `stream_index` for the last frame (synchronises with the labelling). */
BGSB_API int bgsb_pipeline_components(bgsb_pipeline *p, int stream_index, bgsb_component *out, int capacity, int *n);
/* The tables of ALL streams for the last frame into one dense device buffer (one download for the whole group):
 * d_out is int32 [nstreams][(rows_per_stream + 1) * 8]: per stream 8 ints of header {component count, 0 x 7} followed
 * by the first rows_per_stream components (raster order) as bgsb_component rows.  Asynchronous: `stream` (any stream of
 * the device, e.g. the one a download is enqueued on next) waits for the buffer to be complete. */
BGSB_API int bgsb_pipeline_tables_dev(bgsb_pipeline *p, int32_t *d_out, int rows_per_stream, void *stream);
/* cvMoments(pFGMask[R], 0) sums on that stream's cleaned mask, as bgsb_ccl_rect_moments.  BGSB_ERR_ARG when the last
 * frame had the plugin's threshold off and a chain (see bgsb_pipeline_process_dev). */
BGSB_API int bgsb_pipeline_rect_moments(bgsb_pipeline *p, int stream_index, const int32_t *rects_xywh, int nrects,
                                        uint64_t *out);
/* CvBlobDetectorCC::DetectNewBlob for every stream of the last frame, on the labelling the pipeline already ran:
 * bds[s] is stream s's detector (its own lists, tracks and parameters; the same object works with
 * bgsb_blobdetector_detect[_dev] and bgsb_pool_detect), and the results are those of bgsb_blobdetector_detect on the
 * stream's cleaned mask.  One download of all tables, the clustering on the host, ONE moments launch for all streams
 * and one download of the sums: two synchronisations per call whatever nstreams is.
 *   bds[S]         : distinct detectors whose "zeroBorder" is the pipeline's (the masks were labelled with it)
 *   old_blobs[S]   : per stream the tracked blobs (n_old[s] of them; an entry may be NULL when n_old[s] == 0);
 *                    old_blobs == NULL: no stream has any (n_old may then be NULL too)
 *   new_blobs[S]   : stream s's new blob when result[s] == 1
 *   frame_blobs    : nullable, [S][10]: stream s's sorted top-10 (m_pBlobLists[0]), n_frame[s] of them (nullable)
 *   status[S]      : BGSB_OK per stream
 * BGSB_ERR_STATE when the last frame produced no mask (plugin warm-up); BGSB_ERR_ARG for a NULL or repeated detector, a
 * "zeroBorder" mismatch, or the threshold-off-with-chain combination (see bgsb_pipeline_process_dev).  On an error no
 * detector advances. */
BGSB_API int bgsb_pipeline_detect(bgsb_pipeline *p, bgsb_blobdetector *const *bds, const bgsb_blob *const *old_blobs,
                                  const int *n_old, bgsb_blob *new_blobs, int *result, bgsb_blob *frame_blobs,
                                  int *n_frame, int *status);

/* ---------------------------------------------------------------------------------------
 * Stream pool: N camera streams of one geometry over the GPUs of this process (SURVEY 8e; BASELINE configs 4 / 5).
 * The reference's main loop (ustc_src/trackingMain.cpp:161-166; FrameProcessor.cpp:176-195 for the plugin family) serves
 * one camera; the pool runs that loop for many: stream s lives on devices[s % ndevices], each GPU has one host worker
 * thread, one bgsb_pipeline over its streams, and `ring` slots of page-locked frame / mask / table buffers on three CUDA
 * streams, so that slot k+1 uploads while slot k computes and slot k-1 downloads.  Streams never exchange data.
 *   capture side : write frame t of stream s into bgsb_pool_frame_buffer(pool, s, t % ring)   (h*w*3 bytes, dense BGR;
 *                  with "inputFormat" NV12 / I420: h*w*3/2 bytes, the dense 3h/2 x w YUV image)
 *   bgsb_pool_submit(pool, slot, flags)      : every stream's frame of that slot is ready; returns at once
 *   bgsb_pool_wait(pool, slot, &valid)       : that slot's results are on the host; valid = 0 while the plugin warms up
 *   bgsb_pool_mask / bgsb_pool_components    : the cleaned {0,255} mask (if asked for) and the component table
 *                                              (first "tableRows" components in raster order) of one stream
 *   bgsb_pool_detect(pool, slot, ...)        : DetectNewBlob for every stream of the slot (submitted with
 *                                              BGSB_POOL_DETECT), between its wait and its next submit
 * A slot may be refilled and resubmitted once it has been waited for.  One thread drives submit / wait / detect.
 * Submit flags: BGSB_POOL_MASKS downloads the cleaned masks for bgsb_pool_mask; BGSB_POOL_DETECT keeps them on the device
 * for bgsb_pool_detect (one more byte per pixel written, no download; the pipeline's kernel stream then waits for the
 * clean-up and labelling instead of running the next frame set's plugin kernel beside them). 
 * ------------------------------------------------------------------------------------- */
typedef struct bgsb_pool bgsb_pool;
enum { BGSB_POOL_MASKS = 1, BGSB_POOL_DETECT = 2 };
BGSB_API int bgsb_pool_create(bgsb_pool **out, int algo, int nstreams, const int *devices, int ndevices, int w, int h,
                              int ring);
BGSB_API void bgsb_pool_destroy(bgsb_pool *pool);
/* As bgsb_pipeline_set_param / bgsb_pipeline_set_morph, applied to every GPU's pipeline; call before the first submit.
 * The pool's own key "tableRows" (default 256) sets how many components per stream and frame come back to the host.
 * "inputFormat" (BGSB_INPUT_*) is accepted before the first submit only (BGSB_ERR_ARG after it): it resizes the frame
 * buffers and the uploads to h*w*3/2 bytes per stream, and each GPU's pipeline converts its streams' frames. */
BGSB_API int bgsb_pool_set_param(bgsb_pool *pool, const char *key, double value);
BGSB_API int bgsb_pool_set_morph(bgsb_pool *pool, const int *ops, int nops);
BGSB_API int bgsb_pool_device_of(bgsb_pool *pool, int stream, int *device);
BGSB_API int bgsb_pool_info(bgsb_pool *pool, int *ngroups, int *ring, int *table_rows);
BGSB_API uint8_t *bgsb_pool_frame_buffer(bgsb_pool *pool, int stream, int slot);
BGSB_API int bgsb_pool_submit(bgsb_pool *pool, int slot, int flags);
BGSB_API int bgsb_pool_wait(bgsb_pool *pool, int slot, int *valid);
BGSB_API const uint8_t *bgsb_pool_mask(bgsb_pool *pool, int stream, int slot);
BGSB_API int bgsb_pool_components(bgsb_pool *pool, int stream, int slot, bgsb_component *out, int capacity, int *n);
/* bgsb_pipeline_detect for all N streams of a waited-for slot (arguments indexed by global stream id): the clustering
 * on the host from the downloaded tables, then per GPU one moments launch over its streams' masks, all GPUs at once.
 * A stream with more components than "tableRows" gets status[s] = BGSB_ERR_CAPACITY and its detector does not advance;
 * the others complete, and the call returns BGSB_ERR_CAPACITY.  BGSB_ERR_STATE when the slot was not submitted with
 * BGSB_POOL_DETECT, has not been waited for, or holds a warm-up frame. */
BGSB_API int bgsb_pool_detect(bgsb_pool *pool, int slot, bgsb_blobdetector *const *bds, const bgsb_blob *const *old_blobs,
                              const int *n_old, bgsb_blob *new_blobs, int *result, bgsb_blob *frame_blobs, int *n_frame,
                              int *status);

/* ---------------------------------------------------------------------------------------
 * Synthetic video of SURVEY 8(d) generated on the device (bench / tests only):
 * frames [nstreams][T][h][w][3]; stream s uses seed0 + s, frames t0 .. t0+T-1.
 * ------------------------------------------------------------------------------------- */
BGSB_API int bgsb_synth_frames_dev(uint8_t *d_frames, int nstreams, int T, int w, int h,
                                   int t0, uint32_t seed0, void *stream);
/* Mode-churn video: every pixel shows one of five well-separated colours, redrawn every second frame -- the stream
 * on which all K = 5 mixture modes of every pixel stay live (the dense 209 B/px case of SURVEY 8d).  Same layout. */
BGSB_API int bgsb_synth_churn_frames_dev(uint8_t *d_frames, int nstreams, int T, int w, int h,
                                         int t0, uint32_t seed0, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BGSB200_H */
