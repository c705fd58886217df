/*
 * TEST INFRASTRUCTURE ONLY -- CPU restatement (plain C, scalar, one thread) of the
 * foreground-extraction hot path of USTC-Computer-Vision/tracking.
 *
 * It is the parity checker for the CUDA path in tracking_b200/csrc and the "port" CPU
 * baseline of bench.py.  Nothing under tracking_b200/ links, loads or calls it.
 *
 * Where the arithmetic comes from.  The reference's four IBGS plugins
 *   package_bgs/FrameDifferenceBGS.cpp:29-61
 *   package_bgs/AdaptiveBackgroundLearning.cpp:30-83
 *   package_bgs/WeightedMovingVarianceBGS.cpp:30-117,126-138
 *   package_bgs/MixtureOfGaussianV2BGS.cpp:29-74
 * are wrappers over OpenCV calls; OpenCV is an external, un-vendored, un-pinned dependency
 * of the reference (CMakeLists.txt:21 `find_package(OpenCV REQUIRED)`; de-facto 2.4.x).  The
 * per-element semantics of those calls are restated here from OpenCV's published behaviour
 * (modules/video/src/bgfg_gaussmix2.cpp for MOG2, imgproc color/thresh/morph, core arithm)
 * and PINNED against the OpenCV build importable in this image (opencv-python-headless
 * 4.13.0) by tests/test_oracle_pin.py and the golden vectors of tests/golden/ -- see
 * oracle/README.md for the pin status of every function.
 *
 * Build: `make -C oracle` -> oracle/_build/libbgs_oracle.so  (flags keep fp32 unfused).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------ */
/* shared scalar helpers                                                                 */
/* ------------------------------------------------------------------------------------ */

/* cv::cvtColor(CV_BGR2GRAY) on 8UC3, called on the 3-channel DIFFERENCE image at
 * FrameDifferenceBGS.cpp:48, AdaptiveBackgroundLearning.cpp:68, WeightedMovingVarianceBGS.cpp:103.
 * variant 0: OpenCV 4.x 15-bit coefficients; variant 1: OpenCV 2.4 14-bit coefficients
 * (SURVEY.md Appendix B). */
static inline uint8_t gray_bgr(unsigned b, unsigned g, unsigned r, int variant)
{
    if (variant == 0)
        return (uint8_t)((3735u * b + 19235u * g + 9798u * r + 16384u) >> 15);
    return (uint8_t)((1868u * b + 9617u * g + 4899u * r + 8192u) >> 14);
}

/* cv::threshold(src,dst,thr,255,THRESH_BINARY): strict '>' (call sites :51/:71/:106/:62). */
static inline uint8_t thr_u8(uint8_t v, int enable, int thr)
{
    if (!enable) return v;
    return (int)v > thr ? 255 : 0;
}

/* saturate_cast<uchar>(float): cvRound = round-half-to-even, then clamp. */
static inline uint8_t sat_u8_rint(float x)
{
    float r = nearbyintf(x);           /* default rounding mode = to nearest even */
    if (!(r > 0.f)) return 0;          /* also catches NaN like lrint->INT_MIN->0 */
    if (r > 255.f) return 255;
    return (uint8_t)r;
}

ORC_API void orc_gray_bgr(const uint8_t *bgr, int npx, int variant, uint8_t *out)
{
    for (int i = 0; i < npx; i++)
        out[i] = gray_bgr(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2], variant);
}

/* ------------------------------------------------------------------------------------ */
/* FrameDifference  (package_bgs/FrameDifferenceBGS.cpp:45-51)                            */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_fd(const uint8_t *prev, const uint8_t *cur, int npx,
                    int enable_thr, int thr, int gray_variant, uint8_t *fg)
{
    for (int i = 0; i < npx; i++) {
        unsigned d[3];
        for (int c = 0; c < 3; c++) {                       /* cv::absdiff :45 */
            int a = prev[3 * i + c], b = cur[3 * i + c];
            d[c] = (unsigned)(a > b ? a - b : b - a);
        }
        uint8_t g = gray_bgr(d[0], d[1], d[2], gray_variant);   /* :47-48 */
        fg[i] = thr_u8(g, enable_thr, thr);                      /* :50-51 */
    }
}

/* ------------------------------------------------------------------------------------ */
/* StaticFrameDifference (package_bgs/StaticFrameDifferenceBGS.cpp:29-57): the background is   */
/* the first frame, frozen (:34-35); fg = thr(gray(absdiff(in, bg))) (:42-48).                 */
/* Same arithmetic as orc_fd with prev := the frozen background.                               */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_sfd(const uint8_t *bg, const uint8_t *cur, int npx, int enable_thr, int thr,
                     int gray_variant, uint8_t *fg)
{
    orc_fd(bg, cur, npx, enable_thr, thr, gray_variant, fg);
}

/* ------------------------------------------------------------------------------------ */
/* WeightedMovingMean (package_bgs/WeightedMovingMeanBGS.cpp:30-103)                           */
/*   bg_f = 0.5 x0 + 0.3 x1 + 0.2 x2 (:61-62; addWeighted then scaleAdd, as in WMV) or          */
/*          (x0 + x1 + x2)/3.0 (:64): MatExpr lowers it to cv::add(x0,x1) then                   */
/*          addWeighted(t, 1/3., x2, 1/3.) [upstream matop.cpp MatOp_AddEx]                      */
/*   bg8 = sat_u8(rint(bg_f*255)) (:70); fg = thr(gray(absdiff(in, bg8))) (:76-82)               */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_wmm(const uint8_t *cur, const uint8_t *p1, const uint8_t *p2, int npx,
                     int enable_weight, int enable_thr, int thr, int gray_variant, uint8_t *fg, uint8_t *bgout)
{
    const float s = (float)(1. / 255.);
    for (int i = 0; i < npx; i++) {
        unsigned d[3];
        for (int c = 0; c < 3; c++) {
            float x0 = (float)cur[3 * i + c] * s;
            float x1 = (float)p1[3 * i + c] * s;
            float x2 = (float)p2[3 * i + c] * s;
            float m;
            if (enable_weight) {
                float m01 = (float)((double)x0 * 0.5 + (double)x1 * 0.3);
                m = fmaf(x2, (float)0.2, m01);
            } else {
                float t = x0 + x1;
                m = (float)((double)t * (1. / 3.0) + (double)x2 * (1. / 3.0));
            }
            uint8_t b8 = sat_u8_rint(m * 255.f);
            bgout[3 * i + c] = b8;
            int a = cur[3 * i + c];
            d[c] = (unsigned)(a > b8 ? a - b8 : b8 - a);
        }
        fg[i] = thr_u8(gray_bgr(d[0], d[1], d[2], gray_variant), enable_thr, thr);
    }
}

/* ------------------------------------------------------------------------------------ */
/* AdaptiveBackgroundLearning (package_bgs/AdaptiveBackgroundLearning.cpp:43-71)          */
/*   bg is the 8-bit model state (img_background), updated in place and is also the       */
/*   img_bgmodel output (:80).                                                            */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_abl(const uint8_t *in, uint8_t *bg, int npx, double alpha,
                     int enable_thr, int thr, int gray_variant, uint8_t *fg)
{
    const float s = (float)(1. / 255.);                     /* convertTo(CV_32F, 1./255.) :44,47 */
    const double beta = 1 - alpha;                          /* (1-alpha) in double, :54 */
    for (int i = 0; i < npx; i++) {
        unsigned d8[3];
        for (int c = 0; c < 3; c++) {
            float x = (float)in[3 * i + c] * s;
            float y = (float)bg[3 * i + c] * s;
            float d = fabsf(x - y);                          /* absdiff vs OLD bg :49-50 */
            d8[c] = sat_u8_rint(d * 255.f);                  /* :64-65 */
            /* alpha*in_f + (1-alpha)*bg_f -> addWeighted, double accumulate, one cast (A.2) */
            float nb = (float)((double)x * alpha + (double)y * beta);
            bg[3 * i + c] = sat_u8_rint(nb * 255.f);         /* :56-58 */
        }
        uint8_t g = gray_bgr(d8[0], d8[1], d8[2], gray_variant);  /* :67-68 */
        fg[i] = thr_u8(g, enable_thr, thr);                        /* :70-71 */
    }
}

/* ------------------------------------------------------------------------------------ */
/* AdaptiveSelectiveBackgroundLearning (package_bgs/AdaptiveSelectiveBackgroundLearning.cpp:30-105)  */
/*   gray input, 8-bit gray background model `bg` (updated in place), thresholded |in - bg| mask, */
/*   3x3 median (cv::medianBlur replicates the border), then either the adaptive update of every   */
/*   pixel (learning phase, :65-71) or the update of the pixels the mask calls background (:72-90). */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_asbl(const uint8_t *in_bgr, uint8_t *bg, int w, int h, double alpha, int selective,
                      int thr, int gray_variant, uint8_t *fg, uint8_t *scratch /* 2*w*h */)
{
    const float s = (float)(1. / 255.);
    const double beta = 1 - alpha;
    const int npx = w * h;
    uint8_t *gray = scratch, *raw = scratch + npx;
    for (int i = 0; i < npx; i++) {
        gray[i] = gray_bgr(in_bgr[3 * i], in_bgr[3 * i + 1], in_bgr[3 * i + 2], gray_variant);   /* :36-37 */
        float x = (float)gray[i] * s, y = (float)bg[i] * s;                  /* :50-54 */
        float d = fabsf(x - y);                                              /* :56-57 */
        uint8_t d8 = sat_u8_rint(d * 255.f + -0.f);                          /* :59-60 */
        raw[i] = d8 > thr ? 255 : 0;                                         /* :62 */
    }
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {                                        /* :63, BORDER_REPLICATE */
            int cnt = 0;
            for (int dy = -1; dy <= 1; dy++)
                for (int dx = -1; dx <= 1; dx++) {
                    int yy = y + dy < 0 ? 0 : (y + dy >= h ? h - 1 : y + dy);
                    int xx = x + dx < 0 ? 0 : (x + dx >= w ? w - 1 : x + dx);
                    cnt += raw[yy * w + xx] != 0;
                }
            fg[y * w + x] = cnt >= 5 ? 255 : 0;
        }
    for (int i = 0; i < npx; i++) {
        float x = (float)gray[i] * s, y = (float)bg[i] * s;
        float nb = y;
        if (!selective || fg[i] == 0)                                        /* :68 / :82-85 */
            nb = (float)((double)x * alpha + (double)y * beta);
        bg[i] = sat_u8_rint(nb * 255.f + -0.f);                              /* :92-94 */
    }
}

/* ------------------------------------------------------------------------------------ */
/* DPZivkovicAGMMBGS (USTC_BGS type 11): package_bgs/dp/ZivkovicAGMM.cpp:98-372 (SubtractPixel), */
/* called per pixel by Subtract (:382-407); wrapper package_bgs/dp/DPZivkovicAGMMBGS.cpp:32-84.  */
/* The plugin's output is the HIGH-threshold mask (high = 2 * threshold, :60); img_bgmodel is    */
/* never written.  State per pixel: K modes {weight, sigma, mu0, mu1, mu2} + the mode count.     */
/* modes[(i*K + m)*5 + {0 weight, 1 sigma, 2 mu0, 3 mu1, 4 mu2}].  Pinned against a build of the  */
/* reference's own sources (oracle/_ref/libdp_ref.so, `make ref`).                               */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_dpz_apply(const uint8_t *in, int npx, int K, double threshold, double alpha_d,
                           float *modes, uint8_t *nmodes, uint8_t *fg)
{
    const float low_thr = (float)threshold;                   /* params.LowThreshold() = threshold :59 */
    const float high_thr = 2 * low_thr;                       /* :60 */
    const float alpha = (float)alpha_d;                       /* params.Alpha() = alpha :61 (float member) */
    const float bg_threshold = 0.75f, variance = 36.0f, complexity_prior = 0.05f;   /* ZivkovicAGMM.cpp:64-67 */
    for (int i = 0; i < npx; i++) {
        float *md = modes + (size_t)i * K * 5;
        const float p0 = (float)in[3 * i], p1 = (float)in[3 * i + 1], p2 = (float)in[3 * i + 2];
        int fits = 0, bg_high = 0;
        const float one_min_alpha = 1 - alpha;                /* :108 */
        const float prune = -alpha * complexity_prior;        /* :110 */
        int n = nmodes[i];
        float total = 0.0f;
        int bg_gauss = 0;                                     /* :116-128 */
        double sum = 0.0;
        for (int m = 0; m < n; m++) {
            if (sum < bg_threshold) { bg_gauss++; sum += md[m * 5]; }
            else break;
        }
        for (int m = 0; m < n; m++) {                         /* :131-254, n shrinks on prune */
            float *c = md + m * 5;
            float weight = c[0];
            if (!fits) {
                float var = c[1];
                float d0 = c[2] - p0, d1 = c[3] - p1, d2 = c[4] - p2;
                float dist = (d0 * d0 + d1 * d1 + d2 * d2);
                if (dist < high_thr * var && m < bg_gauss) bg_high = 1;            /* :153-154 */
                if (dist < low_thr * var) {                   /* :157 */
                    fits = 1;
                    float k = alpha / weight;                 /* :168, the OLD weight */
                    weight = one_min_alpha * weight + prune;
                    weight += alpha;
                    c[0] = weight;
                    c[2] = c[2] - k * d0; c[3] = c[3] - k * d1; c[4] = c[4] - k * d2;
                    float sigmanew = var + k * (dist - var);  /* :183 */
                    c[1] = sigmanew < 4 ? 4 : sigmanew > 5 * variance ? 5 * variance : sigmanew;   /* :186 */
                    for (int l = m; l > 0; l--) {             /* :212-227 */
                        float *a = md + l * 5, *b = md + (l - 1) * 5;
                        if (a[0] > b[0]) { for (int q = 0; q < 5; q++) { float t = a[q]; a[q] = b[q]; b[q] = t; } }
                        else break;
                    }
                } else {
                    weight = one_min_alpha * weight + prune;  /* :231-238 */
                    if (weight < -prune) { weight = 0.0; n--; }
                    c[0] = weight;
                }
            } else {
                weight = one_min_alpha * weight + prune;      /* :245-252 */
                if (weight < -prune) { weight = 0.0; n--; }
                c[0] = weight;
            }
            total += weight;
        }
        for (int m = 0; m < n; m++) md[m * 5] = md[m * 5] / total;                   /* :257-260 */
        if (!fits) {                                          /* :263-345 */
            if (n != K) n++;
            float *c = md + (n - 1) * 5;
            c[0] = (n == 1) ? 1 : alpha;
            float s2 = 0.0;
            for (int m = 0; m < n; m++) s2 += md[m * 5];
            float inv = 1.0f / s2;
            for (int m = 0; m < n; m++) md[m * 5] *= inv;
            c[2] = p0; c[3] = p1; c[4] = p2; c[1] = variance;
            for (int l = n - 1; l > 0; l--) {
                float *a = md + l * 5, *b = md + (l - 1) * 5;
                if (a[0] > b[0]) { for (int q = 0; q < 5; q++) { float t = a[q]; a[q] = b[q]; b[q] = t; } }
                else break;
            }
        }
        nmodes[i] = (uint8_t)n;
        fg[i] = bg_high ? 0 : 255;                            /* :360-367, Bgs.h:41-42 */
    }
}

/* ------------------------------------------------------------------------------------ */
/* DPAdaptiveMedianBGS / DPMeanBGS / DPWrenGABGS (USTC_BGS types 9, 12, 13): the simple per-pixel models of */
/* the DP package.  Every wrapper (package_bgs/dp/DPAdaptiveMedianBGS.cpp:28-82, DPMeanBGS.cpp:28-84,         */
/* DPWrenGABGS.cpp:28-84) initialises the model from the first frame, then per frame: Subtract -> the HIGH-     */
/* threshold mask is the output (high = 2 * threshold in the parameter class's own type), the low mask is      */
/* cleared, Update() on every pixel.  img_bgmodel is never written.  Pinned against a build of the reference's */
/* own sources (oracle/_ref/libdp_ref.so, `make ref`; tests/golden/golden_dp.json).                            */
/* `first`: no model yet (InitModel from this frame).  frame_num: the wrapper's frameNumber (0 on the first).  */
/* ------------------------------------------------------------------------------------ */
/* AdaptiveMedianBGS.cpp:53-140; thresholds are `unsigned char` members (AdaptiveMedianBGS.h:49-50).            */
ORC_API void orc_dp_median(const uint8_t *in, int npx, int first, int frame_num, int threshold, int sampling_rate,
                           uint8_t *median, uint8_t *fg)
{
    const unsigned char low = (unsigned char)threshold;                      /* DPAdaptiveMedianBGS.cpp:56 */
    const unsigned char high = (unsigned char)(2 * low);                     /* :57 */
    if (first) memcpy(median, in, (size_t)npx * 3);                          /* InitModel :53-63 */
    for (int i = 0; i < npx; i++) {                                          /* SubtractPixel :92-111 */
        int d0 = abs(in[3 * i] - median[3 * i]), d1 = abs(in[3 * i + 1] - median[3 * i + 1]), d2 = abs(in[3 * i + 2] - median[3 * i + 2]);
        fg[i] = (d0 <= high && d1 <= high && d2 <= high) ? 0 : 255;
    }
    if (frame_num % sampling_rate == 1) {                                    /* Update :65-90, mask cleared: every pixel */
        for (int i = 0; i < npx * 3; i++) {
            if (in[i] > median[i]) median[i]++;
            else if (in[i] < median[i]) median[i]--;
        }
    }
}

/* MeanBGS.cpp:32-131; thresholds are `unsigned int` members, alpha is a float member (MeanBGS.h:47-62).        */
ORC_API void orc_dp_mean(const uint8_t *in, int npx, int first, int threshold, double alpha_d, float *mean, uint8_t *fg)
{
    const unsigned int low = (unsigned int)threshold;                        /* DPMeanBGS.cpp:56 */
    const unsigned int high = 2 * low;                                       /* :57 */
    const float alpha = (float)alpha_d;                                      /* :59 */
    if (first) for (int i = 0; i < npx * 3; i++) mean[i] = (float)in[i];     /* InitModel :40-52 */
    for (int i = 0; i < npx; i++) {                                          /* SubtractPixel :77-99 */
        float dist = 0;
        for (int ch = 0; ch < 3; ch++) dist += (in[3 * i + ch] - mean[3 * i + ch]) * (in[3 * i + ch] - mean[3 * i + ch]);
        fg[i] = dist > high ? 255 : 0;
    }
    for (int i = 0; i < npx * 3; i++)                                        /* Update :54-75 */
        mean[i] = alpha * mean[i] + (1.0f - alpha) * in[i];
}

/* WrenGA.cpp:47-173; thresholds and alpha are float members (WrenGA.h:48-62); one variance per pixel (var[0]). */
/* state[4 * i + {0, 1, 2}] = mu, state[4 * i + 3] = var[0].                                                    */
ORC_API void orc_dp_wren(const uint8_t *in, int npx, int first, double threshold, double alpha_d, float *state, uint8_t *fg)
{
    const float low = (float)threshold;                                      /* DPWrenGABGS.cpp:56 */
    const float high = 2 * low;                                              /* :57 */
    const float alpha = (float)alpha_d;                                      /* :58 */
    const float variance = 36.0f;                                            /* WrenGA.cpp:51 */
    (void)low;
    if (first)                                                               /* InitModel :67-85 */
        for (int i = 0; i < npx; i++) {
            for (int ch = 0; ch < 3; ch++) state[4 * i + ch] = in[3 * i + ch];
            state[4 * i + 3] = variance;
        }
    for (int i = 0; i < npx; i++) {
        float *g = state + 4 * (size_t)i;
        float dist = 0;                                                      /* SubtractPixel :121-147 */
        for (int ch = 0; ch < 3; ch++) { float delta = g[ch] - in[3 * i + ch]; dist += delta * delta; }
        fg[i] = dist > high * g[3] ? 255 : 0;
    }
    for (int i = 0; i < npx; i++) {                                          /* Update :87-119 */
        float *g = state + 4 * (size_t)i;
        float dR = g[0] - in[3 * i], dG = g[1] - in[3 * i + 1], dB = g[2] - in[3 * i + 2];
        float dist = (dR * dR + dG * dG + dB * dB);
        g[0] -= alpha * (dR); g[1] -= alpha * (dG); g[2] -= alpha * (dB);
        float sigmanew = g[3] + alpha * (dist - g[3]);
        g[3] = sigmanew < 4 ? 4 : sigmanew > 5 * variance ? 5 * variance : sigmanew;
    }
}

/* ------------------------------------------------------------------------------------ */
/* DPPratiMediodBGS (USTC_BGS type 14): package_bgs/dp/PratiMediodBGS.cpp:52-275, wrapper DPPratiMediodBGS.cpp:28-88.  */
/* Pure integer.  Per pixel a circular buffer of up to H sampled pixels with, for every sample, the sum of its L-inf   */
/* distances to the other samples; the medoid (smallest sum, first wins) is the background.  Because the wrapper       */
/* clears the update mask, every pixel is updated on every sampled frame, so the buffer length n and the write         */
/* position pos are the same for all pixels: samples[s] (s < n) are whole frames, dist[s] whole int planes.            */
/* Per frame (wrapper :66-68): Subtract with the medoid as it stands, then Update.                                     */
/* The quirks are the reference's: when the buffer is full the sample being replaced still takes part in the medoid    */
/* search with its old sum (:99-117 subtracts its distances from the OTHERS, UpdateMediod :128-165 then walks over     */
/* all H samples), and the new sample's sum includes its distance to the one it replaces.  `weight` is never used.     */
/* ------------------------------------------------------------------------------------ */
static int orc_linf(const uint8_t *a, const uint8_t *b)
{
    int m = 0;
    for (int ch = 0; ch < 3; ch++) { int d = abs(a[ch] - b[ch]); if (d > m) m = d; }
    return m;
}

/* Subtract :236-262 + CalculateMasks :204-234 + Combine :167-202; fg = the combined mask (both outputs are the same) */
ORC_API void orc_dp_prati_subtract(const uint8_t *in, int w, int h, int frame_num, int threshold, int history_size,
                                   const uint8_t *median, uint8_t *fg, uint8_t *scratch /* 2 * w * h */)
{
    const unsigned int low = (unsigned int)threshold, high = 2 * low;        /* DPPratiMediodBGS.cpp:57-58, unsigned int members */
    const int npx = w * h;
    memset(fg, 0, (size_t)npx);
    if (frame_num < history_size) return;                                    /* :239-244 */
    uint8_t *lo = scratch, *hi = scratch + npx;
    for (int i = 0; i < npx; i++) {
        unsigned char dist = (unsigned char)orc_linf(in + 3 * i, median + 3 * i);
        lo[i] = dist > low ? 255 : 0;
        hi[i] = dist > high ? 255 : 0;
    }
    for (int r = 1; r < h - 1; r++)                                          /* the image border stays BACKGROUND :175-176 */
        for (int c = 1; c < w - 1; c++) {
            const int i = r * w + c;
            if (hi[i]) fg[i] = 255;
            else if (lo[i]) {
                int any = 0;
                for (int dr = -1; dr <= 1; dr++) for (int dc = -1; dc <= 1; dc++) if (dr || dc) any |= hi[i + dr * w + dc];
                if (any) fg[i] = 255;
            }
        }
}

/* Update :70-126 + UpdateMediod :128-165 for a sampled frame (the caller checks frame_num % samplingRate == 0).       */
/* samples: [H][npx * 3], dist: [H][npx], n = samples held so far (all pixels alike), pos = the slot to replace once   */
/* n == H; median: [npx * 3].  The caller advances n / pos afterwards.                                                 */
ORC_API void orc_dp_prati_update(const uint8_t *in, int npx, int n, int pos, int history_size, uint8_t *samples, int32_t *dist,
                                 uint8_t *median)
{
    const size_t fb = (size_t)npx * 3;
    const int full = n == history_size;
    for (int i = 0; i < npx; i++) {
        const uint8_t *px = in + 3 * (size_t)i;
        if (full) {                                                          /* :84-95 */
            const uint8_t *old = samples + pos * fb + 3 * (size_t)i;
            for (int s = 0; s < n; s++) dist[(size_t)s * npx + i] -= orc_linf(old, samples + s * fb + 3 * (size_t)i);
        }
        int median_dist = 2147483647, L = 0;                                 /* UpdateMediod */
        uint8_t med[3] = {median[3 * i], median[3 * i + 1], median[3 * i + 2]};
        for (int s = 0; s < n; s++) {
            const uint8_t *sp = samples + s * fb + 3 * (size_t)i;
            const int d = orc_linf(sp, px);
            int32_t *ds = dist + (size_t)s * npx + i;
            *ds += d;
            if (*ds < median_dist) { median_dist = *ds; med[0] = sp[0]; med[1] = sp[1]; med[2] = sp[2]; }
            L += d;
        }
        if (L < median_dist) { med[0] = px[0]; med[1] = px[1]; med[2] = px[2]; }
        median[3 * i] = med[0]; median[3 * i + 1] = med[1]; median[3 * i + 2] = med[2];
        const int slot = full ? pos : n;                                     /* :97-100 / :119-121 */
        dist[(size_t)slot * npx + i] = L;
        uint8_t *dst = samples + slot * fb + 3 * (size_t)i;
        dst[0] = px[0]; dst[1] = px[1]; dst[2] = px[2];
    }
}

/* ------------------------------------------------------------------------------------ */
/* SigmaDeltaBGS (USTC_BGS type 35): package_bgs/bl/sdLaMa091.cpp:117-232 (init), :470-636 (update), wrapper          */
/* package_bgs/bl/SigmaDeltaBGS.cpp:21-50.  Pure integer, per byte of the interleaved BGR row:                        */
/*   Mt moves one step towards the pixel; Ot = absVal((int8_t)(Mt - I)) -- the difference passes through a signed     */
/*   char, so |d| > 128 wraps (:74-76, :559); Vt moves one step towards N * Ot in uint8_t arithmetic (it wraps) and   */
/*   is clamped by the uint8_t min / max helpers to the parameters truncated to a byte (:62-63, :574-584); a pixel    */
/*   is foreground when Ot >= Vt in any channel (:604-624).  The first frame only initialises: Mt = frame, Vt = Vmin  */
/*   for the first `width` BYTES of every row and -- the C3R initialiser delegates to the C1R one -- nothing for the  */
/*   rest, taken as zero here (oracle/ref_dp/sd_ref.cpp says why).  Parameters are applied before every frame.        */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_sigma_delta(const uint8_t *in, int w, int h, int first, int amp, int min_var, int max_var,
                             uint8_t *Mt, uint8_t *Vt, uint8_t *fg)
{
    const size_t nb = (size_t)w * h * 3;
    const uint32_t N = (uint32_t)amp, Vmin = (uint32_t)min_var, Vmax = (uint32_t)max_var;
    if (first) {
        memcpy(Mt, in, nb);                                                   /* :155 */
        for (int r = 0; r < h; r++)                                           /* :204-216 with width, not rgbWidth */
            for (int j = 0; j < 3 * w; j++) Vt[(size_t)r * 3 * w + j] = j < w ? (uint8_t)Vmin : 0;
        return;
    }
    for (size_t i = 0; i < nb; i += 3) {
        int fgpx = 0;
        for (int ch = 0; ch < 3; ch++) {
            uint8_t m = Mt[i + ch], v = Vt[i + ch];
            const uint8_t x = in[i + ch];
            if (m < x) ++m; else if (m > x) --m;                             /* :536-539 */
            Mt[i + ch] = m;
            const int8_t d8 = (int8_t)(m - x);                                /* absVal's parameter type */
            const uint8_t o = d8 < 0 ? (uint8_t)-d8 : (uint8_t)d8;            /* :74-76 */
            const uint32_t amp_o = N * o;                                     /* :574 */
            if (v < amp_o) ++v; else if (v > amp_o) --v;                      /* :576-579, uint8_t */
            const uint8_t lo = v < (uint8_t)Vmax ? v : (uint8_t)Vmax;         /* min(uint8_t, uint8_t) :581 */
            v = lo > (uint8_t)Vmin ? lo : (uint8_t)Vmin;
            Vt[i + ch] = v;
            if (o >= v) fgpx = 1;                                             /* :604-605 */
        }
        fg[i / 3] = fgpx ? 255 : 0;
    }
}

/* ------------------------------------------------------------------------------------ */
/* WeightedMovingVariance (package_bgs/WeightedMovingVarianceBGS.cpp:53-106,126-138)       */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_wmv(const uint8_t *cur, const uint8_t *p1, const uint8_t *p2, int npx,
                     int enable_weight, int enable_thr, int thr, int gray_variant, uint8_t *fg)
{
    const float s = (float)(1. / 255.);
    const double w0 = enable_weight ? 0.5 : 0.3, w1 = 0.3, w2 = enable_weight ? 0.2 : 0.3;  /* :66-70 */
    const float w0f = (float)w0, w1f = (float)w1, w2f = (float)w2;
    for (int i = 0; i < npx; i++) {
        unsigned g8[3];
        for (int c = 0; c < 3; c++) {
            float x0 = (float)cur[3 * i + c] * s;
            float x1 = (float)p1[3 * i + c] * s;
            float x2 = (float)p2[3 * i + c] * s;
            /* (A*w0 + B*w1) -> addWeighted (double), + C*w2 -> scaleAdd (fused) :67-70 */
            float m01 = (float)((double)x0 * w0 + (double)x1 * w1);
            float m = fmaf(x2, w2f, m01);
            /* computeWeightedVariance :126-138 : absdiff, pow 2 (= x*x), weight*Mat (fp32 mul) */
            float d0 = fabsf(x0 - m), d1 = fabsf(x1 - m), d2 = fabsf(x2 - m);
            float v0 = (d0 * d0) * w0f, v1 = (d1 * d1) * w1f, v2 = (d2 * d2) * w2f;
            float v = (v0 + v1) + v2;                        /* :84 left-assoc MatExpr sum */
            float sd = sqrtf(v);                             /* :95 */
            g8[c] = sat_u8_rint(sd * 255.f);                 /* :99 */
        }
        uint8_t g = gray_bgr(g8[0], g8[1], g8[2], gray_variant);  /* :102-103 */
        fg[i] = thr_u8(g, enable_thr, thr);                        /* :105-106 */
    }
}

/* ------------------------------------------------------------------------------------ */
/* MOG2: cv::BackgroundSubtractorMOG2::operator() + getBackgroundImage                    */
/*   (member `mog`, package_bgs/MixtureOfGaussianV2BGS.h:30; calls .cpp:56,59).           */
/*   State layout here follows upstream (AoS): gmm[npx][K]{weight,variance},               */
/*   mean[npx][K][3], nmodes[npx].  SURVEY.md Appendix A.4 is the spec.                    */
/* ------------------------------------------------------------------------------------ */
typedef struct {
    int   K;            /* nmixtures, 5 */
    float Tb;           /* varThreshold 16 */
    float Tg;           /* varThresholdGen 9 */
    float TB;           /* backgroundRatio 0.9 */
    float varInit, varMin, varMax;   /* 15, 4, 75 */
    float CT;           /* complexity reduction 0.05 */
    float tau;          /* shadow threshold 0.5 */
    int   detect_shadows;   /* 1 */
    int   shadow_value;     /* 127 */
    int   history;          /* 500 */
} orc_mog2_params;

ORC_API void orc_mog2_default_params(orc_mog2_params *p)
{
    p->K = 5; p->Tb = 16.f; p->Tg = 9.f; p->TB = 0.9f;
    p->varInit = 15.f; p->varMin = 4.f; p->varMax = 75.f;
    p->CT = 0.05f; p->tau = 0.5f; p->detect_shadows = 1; p->shadow_value = 127; p->history = 500;
}

/* learning rate rule of operator(): ++nframes;
 * lr = (alpha >= 0 && nframes > 1) ? alpha : 1./min(2*nframes, history).
 * alpha >= 1 re-initialises the model first (needToInitialize, nframes = 0): the caller then passes nframes 1. */
ORC_API double orc_mog2_learning_rate(double alpha, int nframes_after_increment, int history)
{
    if (alpha >= 0 && nframes_after_increment > 1) return alpha;
    int d = 2 * nframes_after_increment; if (d > history) d = history;
    return 1. / d;
}

static int mog2_shadow(const float *d, int n, const float *gmm, const float *mean,
                       const orc_mog2_params *P)
{
    float tW = 0.f;
    for (int m = 0; m < n; m++) {
        const float *mu = mean + 3 * m;
        float num = 0.f, den = 0.f;
        for (int c = 0; c < 3; c++) { num += d[c] * mu[c]; den += mu[c] * mu[c]; }
        if (den == 0.f) return 0;
        if (num <= den && num >= P->tau * den) {
            float a = num / den, e = 0.f;
            for (int c = 0; c < 3; c++) { float dd = a * mu[c] - d[c]; e += dd * dd; }
            if (e < P->Tb * gmm[2 * m + 1] * a * a) return 1;
        }
        tW += gmm[2 * m];
        if (tW > P->TB) return 0;
    }
    return 0;
}

static inline void swap_mode(float *gmm, float *mean, int i, int j)
{
    float t;
    t = gmm[2 * i]; gmm[2 * i] = gmm[2 * j]; gmm[2 * j] = t;
    t = gmm[2 * i + 1]; gmm[2 * i + 1] = gmm[2 * j + 1]; gmm[2 * j + 1] = t;
    for (int c = 0; c < 3; c++) { t = mean[3 * i + c]; mean[3 * i + c] = mean[3 * j + c]; mean[3 * j + c] = t; }
}

/* One frame.  lr is the already-resolved learning rate (see orc_mog2_learning_rate).
 * mask receives the RAW MOG2 output {0, shadow_value, 255}. */
ORC_API void orc_mog2_apply(const uint8_t *in, int npx, double lr, const orc_mog2_params *P,
                            float *gmm_all, float *mean_all, uint8_t *nmodes_all, uint8_t *mask)
{
    const int K = P->K;
    const float alphaT = (float)lr, alpha1 = 1.f - alphaT;
    const float prune = (float)(-lr * (double)P->CT);   /* float prune = -learningRate*fCT (fCT float, product in double) */
    /* MOG2Invoker: varMin = min(_varMin, _varMax), varMax = max(_varMin, _varMax) */
    const float varMin = P->varMin < P->varMax ? P->varMin : P->varMax;
    const float varMax = P->varMin < P->varMax ? P->varMax : P->varMin;
    for (int i = 0; i < npx; i++) {
        float *gmm = gmm_all + (size_t)i * K * 2;
        float *mean = mean_all + (size_t)i * K * 3;
        float d[3] = { (float)in[3 * i], (float)in[3 * i + 1], (float)in[3 * i + 2] };
        int n = nmodes_all[i];
        int bg = 0, fits = 0;
        float tw = 0.f;
        for (int m = 0; m < n; m++) {           /* bound is the LIVE n (A.4 loop-bound note) */
            float w = alpha1 * gmm[2 * m] + prune;
            int swaps = 0;
            if (!fits) {
                float *mu = mean + 3 * m;
                float var = gmm[2 * m + 1];
                float dD0 = mu[0] - d[0], dD1 = mu[1] - d[1], dD2 = mu[2] - d[2];
                float dist2 = dD0 * dD0 + dD1 * dD1 + dD2 * dD2;
                if (tw < P->TB && dist2 < P->Tb * var) bg = 1;
                if (dist2 < P->Tg * var) {
                    fits = 1;
                    w += alphaT;
                    float k = alphaT / w;
                    mu[0] -= k * dD0; mu[1] -= k * dD1; mu[2] -= k * dD2;
                    float vn = var + k * (dist2 - var);
                    vn = vn > varMin ? vn : varMin;             /* MAX(varnew, varMin) */
                    vn = vn < varMax ? vn : varMax;             /* MIN(varnew, varMax) */
                    gmm[2 * m + 1] = vn;
                    for (int j = m; j > 0; j--) {
                        if (w < gmm[2 * (j - 1)]) break;
                        swaps++;
                        swap_mode(gmm, mean, j, j - 1);
                    }
                }
            }
            if (w < -prune) { w = 0.f; n--; }
            gmm[2 * (m - swaps)] = w;
            tw += w;
        }
        /* renormalise (4.x guards |tw| > FLT_EPSILON; with n>0 tw >= -prune so identical) */
        float inv = 0.f;
        if (fabsf(tw) > 1.1920929e-07f) inv = 1.f / tw;
        for (int m = 0; m < n; m++) gmm[2 * m] *= inv;
        if (!fits && alphaT > 0.f) {
            int m = (n == K) ? K - 1 : n++;
            if (n == 1) gmm[2 * m] = 1.f;
            else {
                gmm[2 * m] = alphaT;
                for (int j = 0; j < n - 1; j++) gmm[2 * j] *= alpha1;
            }
            mean[3 * m] = d[0]; mean[3 * m + 1] = d[1]; mean[3 * m + 2] = d[2];
            gmm[2 * m + 1] = P->varInit;
            for (int j = n - 1; j > 0; j--) {
                if (alphaT < gmm[2 * (j - 1)]) break;
                swap_mode(gmm, mean, j, j - 1);
            }
        }
        nmodes_all[i] = (uint8_t)n;
        mask[i] = bg ? 0 : ((P->detect_shadows && mog2_shadow(d, n, gmm, mean, P)) ? (uint8_t)P->shadow_value : 255);
    }
}

/* getBackgroundImage (MixtureOfGaussianV2BGS.cpp:59). */
ORC_API void orc_mog2_background(int npx, const orc_mog2_params *P, const float *gmm_all,
                                 const float *mean_all, const uint8_t *nmodes_all, uint8_t *bgimg)
{
    const int K = P->K;
    for (int i = 0; i < npx; i++) {
        const float *gmm = gmm_all + (size_t)i * K * 2;
        const float *mean = mean_all + (size_t)i * K * 3;
        int n = nmodes_all[i];
        float acc[3] = { 0.f, 0.f, 0.f }, tw = 0.f;
        for (int m = 0; m < n; m++) {
            float w = gmm[2 * m];
            for (int c = 0; c < 3; c++) acc[c] += w * mean[3 * m + c];
            tw += w;
            if (tw > P->TB) break;
        }
        float inv = 0.f;
        if (fabsf(tw) > 1.1920929e-07f) inv = 1.f / tw;
        for (int c = 0; c < 3; c++) bgimg[3 * i + c] = sat_u8_rint(acc[c] * inv);
    }
}

/* ------------------------------------------------------------------------------------ */
/* Morphology: cv::erode / cv::dilate with the default 3x3 rect element, anchor centre,    */
/* out-of-image pixels ignored (SURVEY.md A.5).  op: 0 erode, 1 dilate.                    */
/* ------------------------------------------------------------------------------------ */
ORC_API void orc_morph3x3(const uint8_t *in, int w, int h, int op, int iterations, uint8_t *out)
{
    size_t n = (size_t)w * h;
    uint8_t *a = (uint8_t *)malloc(n), *b = (uint8_t *)malloc(n);
    memcpy(a, in, n);
    for (int it = 0; it < iterations; it++) {
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                int v = op ? 0 : 255;
                for (int dy = -1; dy <= 1; dy++) {
                    int yy = y + dy; if (yy < 0 || yy >= h) continue;
                    for (int dx = -1; dx <= 1; dx++) {
                        int xx = x + dx; if (xx < 0 || xx >= w) continue;
                        int p = a[(size_t)yy * w + xx];
                        if (op) { if (p > v) v = p; } else { if (p < v) v = p; }
                    }
                }
                b[(size_t)y * w + x] = (uint8_t)v;
            }
        uint8_t *t = a; a = b; b = t;
    }
    memcpy(out, a, n);
    free(a); free(b);
}

/* ------------------------------------------------------------------------------------ */
/* Connected components: steps 1-2 of CvBlobDetectorCC::DetectNewBlob (SURVEY.md A.6).     */
/*   foreground = mask > 128; 8-connectivity; canonical label k (1-based) = rank of the    */
/*   component's minimum linear index.  Plain BFS flood fill in raster order, which         */
/*   numbers components by raster-first pixel by construction.                              */
/*   zero_border: emulate OpenCV<=3.1 cvFindContours, which clears the outer 1-px frame.    */
/*   external[k-1] = 1 iff the component is NOT enclosed in a hole of another component     */
/*   (what RETR_EXTERNAL keeps): its surrounding background region (4-connected) reaches    */
/*   the outside of the image.                                                              */
/*   stats[k-1] = {xmin, ymin, xmax, ymax, area, first_linear_index}                        */
/* ------------------------------------------------------------------------------------ */
ORC_API int orc_ccl8(const uint8_t *mask, int w, int h, int zero_border,
                     int32_t *labels, int max_comp, int32_t *stats, uint8_t *external)
{
    size_t n = (size_t)w * h;
    uint8_t *fgm = (uint8_t *)malloc(n);
    for (size_t i = 0; i < n; i++) fgm[i] = mask[i] > 128;
    if (zero_border) {
        for (int x = 0; x < w; x++) { fgm[x] = 0; fgm[(size_t)(h - 1) * w + x] = 0; }
        for (int y = 0; y < h; y++) { fgm[(size_t)y * w] = 0; fgm[(size_t)y * w + w - 1] = 0; }
    }
    memset(labels, 0, n * sizeof(int32_t));
    int32_t *queue = (int32_t *)malloc(n * sizeof(int32_t));
    int ncomp = 0;
    for (size_t p0 = 0; p0 < n; p0++) {
        if (!fgm[p0] || labels[p0]) continue;
        ncomp++;
        int xmin = w, ymin = h, xmax = -1, ymax = -1, area = 0;
        size_t qh = 0, qt = 0;
        queue[qt++] = (int32_t)p0; labels[p0] = ncomp;
        while (qh < qt) {
            int p = queue[qh++];
            int x = p % w, y = p / w;
            area++;
            if (x < xmin) xmin = x; if (x > xmax) xmax = x;
            if (y < ymin) ymin = y; if (y > ymax) ymax = y;
            for (int dy = -1; dy <= 1; dy++) {
                int yy = y + dy; if (yy < 0 || yy >= h) continue;
                for (int dx = -1; dx <= 1; dx++) {
                    int xx = x + dx; if (xx < 0 || xx >= w) continue;
                    size_t q = (size_t)yy * w + xx;
                    if (fgm[q] && !labels[q]) { labels[q] = ncomp; queue[qt++] = (int32_t)q; }
                }
            }
        }
        if (ncomp <= max_comp && stats) {
            int32_t *s = stats + 6 * (size_t)(ncomp - 1);
            s[0] = xmin; s[1] = ymin; s[2] = xmax; s[3] = ymax; s[4] = area; s[5] = (int32_t)p0;
        }
    }
    if (external) {
        /* flood the background (4-connected) from outside the image */
        uint8_t *outer = (uint8_t *)calloc(n, 1);
        size_t qh = 0, qt = 0;
        for (int x = 0; x < w; x++) {
            size_t a = x, b = (size_t)(h - 1) * w + x;
            if (!fgm[a] && !outer[a]) { outer[a] = 1; queue[qt++] = (int32_t)a; }
            if (!fgm[b] && !outer[b]) { outer[b] = 1; queue[qt++] = (int32_t)b; }
        }
        for (int y = 0; y < h; y++) {
            size_t a = (size_t)y * w, b = (size_t)y * w + w - 1;
            if (!fgm[a] && !outer[a]) { outer[a] = 1; queue[qt++] = (int32_t)a; }
            if (!fgm[b] && !outer[b]) { outer[b] = 1; queue[qt++] = (int32_t)b; }
        }
        static const int d4x[4] = { 1, -1, 0, 0 }, d4y[4] = { 0, 0, 1, -1 };
        while (qh < qt) {
            int p = queue[qh++];
            int x = p % w, y = p / w;
            for (int k = 0; k < 4; k++) {
                int xx = x + d4x[k], yy = y + d4y[k];
                if (xx < 0 || xx >= w || yy < 0 || yy >= h) continue;
                size_t q = (size_t)yy * w + xx;
                if (!fgm[q] && !outer[q]) { outer[q] = 1; queue[qt++] = (int32_t)q; }
            }
        }
        int lim = ncomp < max_comp ? ncomp : max_comp;
        for (int k = 0; k < lim; k++) {
            int p0 = stats[6 * (size_t)k + 5];
            int x = p0 % w;
            /* the pixel left of the raster-first pixel lies in the surrounding background */
            external[k] = (x == 0) ? 1 : outer[p0 - 1];
        }
        free(outer);
    }
    free(queue); free(fgm);
    return ncomp;
}

/* cvMoments(pFG[R], binary=0) on an 8-bit ROI: raw spatial moments up to order 2 that
 * CvBlobDetectorCC uses (step 4 of A.6): m00 m10 m01 m20 m02 (+ m11), pixel-VALUE weighted,
 * x,y relative to the ROI origin.  Exact integer sums. */
ORC_API void orc_rect_moments(const uint8_t *img, int w, int h, int rx, int ry, int rw, int rh,
                              uint64_t out[6])
{
    uint64_t m00 = 0, m10 = 0, m01 = 0, m20 = 0, m02 = 0, m11 = 0;
    (void)h;
    for (int y = 0; y < rh; y++)
        for (int x = 0; x < rw; x++) {
            uint64_t v = img[(size_t)(ry + y) * w + rx + x];
            m00 += v; m10 += v * x; m01 += v * y; m20 += v * x * x; m02 += v * y * y; m11 += v * x * y;
        }
    out[0] = m00; out[1] = m10; out[2] = m01; out[3] = m20; out[4] = m02; out[5] = m11;
}

/* ------------------------------------------------------------------------------------ */
/* Synthetic video of SURVEY.md 8(d) (integer-only, so CPU and GPU generate identical      */
/* frames).  Used by the CPU baseline legs so the generator is not timed in Python.         */
/* ------------------------------------------------------------------------------------ */
static inline uint32_t mix32(uint32_t h)
{
    h ^= h >> 16; h *= 0x7feb352dU; h ^= h >> 15; h *= 0x846ca68bU; h ^= h >> 16;
    return h;
}

ORC_API void orc_synth_frame(int w, int h, int t, uint32_t seed, uint8_t *bgr)
{
    const int scale = (w >= 3840) ? 2 : 1;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            for (int c = 0; c < 3; c++) {
                int B = 32 + (((x * 5 + y * 3 + 64 * c) >> 3) & 127) + 48 * (((x >> 6) ^ (y >> 6)) & 1);
                uint32_t hsh = ((uint32_t)x * 73856093U) ^ ((uint32_t)y * 19349663U) ^
                               ((uint32_t)t * 83492791U) ^ ((uint32_t)c * 2654435761U) ^ seed;
                int N = (int)(mix32(hsh) % 13U) - 6;
                int v = B + N; if (v < 0) v = 0; if (v > 255) v = 255;
                bgr[((size_t)y * w + x) * 3 + c] = (uint8_t)v;
            }
    for (int r = 0; r < 12; r++) {
        int rw = 100 * scale, rh = 80 * scale;
        int x0 = (100 + 150 * r + 17 * t) % (w - 120 * scale);
        int y0 = (60 + 83 * r + 5 * t) % (h - 90 * scale);
        uint8_t col[3] = { (uint8_t)((40 * r) & 255), (uint8_t)(255 - 20 * r), 128 };
        for (int y = y0; y < y0 + rh && y < h; y++)
            for (int x = x0; x < x0 + rw && x < w; x++)
                for (int c = 0; c < 3; c++) bgr[((size_t)y * w + x) * 3 + c] = col[c];
    }
}

/* Mode-churn video (tracking_b200/csrc/synth.cu: synth_churn_kernel): five colours per pixel, redrawn every 2nd frame. */
ORC_API void orc_synth_churn_frame(int w, int h, int t, uint32_t seed, uint8_t *bgr)
{
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            uint32_t hi = ((uint32_t)x * 73856093U) ^ ((uint32_t)y * 19349663U) ^ ((uint32_t)(t >> 1) * 83492791U) ^ (seed * 2246822519U);
            int i = (int)(mix32(hi) % 5U);
            int col[3] = { 20 + 50 * i, 230 - 45 * i, (90 + 110 * i) & 255 };
            for (int c = 0; c < 3; c++) {
                uint32_t hsh = ((uint32_t)x * 73856093U) ^ ((uint32_t)y * 19349663U) ^
                               ((uint32_t)t * 83492791U) ^ ((uint32_t)c * 2654435761U) ^ seed;
                int v = col[c] + (int)(mix32(hsh) % 5U) - 2;
                if (v < 0) v = 0; if (v > 255) v = 255;
                bgr[((size_t)y * w + x) * 3 + c] = (uint8_t)v;
            }
        }
}
