// Internal launch descriptors shared between the C-ABI layer (capi.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bgsb {

// ---- FD / ABL / WMV ---------------------------------------------------------------------------
struct SimpleLaunch {
    const uint8_t *frames;   // [S][T][npx*3]
    uint8_t *fg;             // [S][T][npx]
    uint8_t *bg;             // ABL only: [S][T][npx*3] or [S][npx*3] (bg_last_only), nullable
    const uint8_t *hist0;    // read : FD prev / WMV prev_1 / ABL 8-bit background   [S][npx*3]
    const uint8_t *hist1;    // read : WMV prev_2
    uint8_t *hist0_out;      // write-back targets (nullable = history lives in caller-visible ring)
    uint8_t *hist1_out;
    int npx, T;
    int have_hist;           // how many history images are valid on entry (0,1,2)
    int bg_last_only;
    int enable_thr, thr, gray_variant;
    double alpha;            // ABL
    int abl_update;          // ABL: limit == -1 (AdaptiveBackgroundLearning.cpp:52); 0 freezes the model
    const uint8_t *abl_lut;  // ABL: 64 KB table of the blend for this alpha (abl_lut_index), null = arithmetic kernel
    int abl_lut_mode;        // ABL table kernels: 0 = warp-coalesced where the alignment allows, 1 = per-thread groups
    int abl_quiet;           // ABL, warp-coalesced kernel: use the table's quiet radius (stored behind the table) to skip lookups
    double w0, w1, w2;       // WMV weights (0.5,0.3,0.2 | 0.3,0.3,0.3)
    int quiet_range;         // WMV, thresholded output: a 16-pixel group whose 48 bytes each moved by at most this much over the
                             // three frames has an all-zero mask (launch_wmv_bound_table proves it); -1 = no shortcut
    float one;               // 1.0f at run time: keeps ptxas from contracting packed mul + add (mog2_fastmath.cuh)
};
int launch_simple(int algo, const SimpleLaunch &L, int nstreams, cudaStream_t stream);
// WMV: d_table[r] (256 unsigned, zeroed by the callee) = the largest re-quantised standard deviation byte over ALL byte
// triples (b0, b1, b2) with max - min == r, computed with the kernel's own per-channel routine for these weights.
int launch_wmv_bound_table(unsigned *d_table, double w0, double w1, double w2, cudaStream_t stream);
// Fill the 64 KB ABL table for `alpha` with the arithmetic kernel's own blend (bit-exact by construction).
// blend_variant 0: OpenCV 4.x double-precision addWeighted (pinned); 1: OpenCV 2.4 fp32 addWeighted (unpinned).
// the 64 KB byte-pair table plus the int that holds its quiet radius (abl_lut_radius_kernel)
#define ABL_LUT_BYTES (65536 + 256)
int launch_abl_lut_build(uint8_t *d_lut, double alpha, int blend_variant, cudaStream_t stream);

// ---- AdaptiveSelectiveBackgroundLearning (single-channel model; one frame per launch pair) --------
struct AsblLaunch {
    const uint8_t *frame;    // [S] BGR frames, frame_stride bytes apart
    uint8_t *fg;             // [S] masks, fg_stride bytes apart
    uint8_t *bgout;          // [S] gray background images, bg_stride bytes apart, nullable
    uint8_t *model;          // [S][npx] 8-bit gray background model
    uint8_t *model_out;      // [S][npx] second model buffer: the single-pass kernel reads `model` and writes this one
    uint8_t *gray, *raw;     // [S][npx] scratch: gray input, thresholded difference before the median
    size_t frame_stride, fg_stride, bg_stride;
    int w, h;
    int first;               // no model yet: it starts as the gray input (AdaptiveSelectiveBackgroundLearning.cpp:47-48)
    int selective;           // 0: learning phase, every pixel is blended (:65-71); 1: only background pixels (:72-90)
    double alpha;            // alphaLearn or alphaDetection
    const uint8_t *lut;      // 64 KB blend table for alpha (launch_abl_lut_build): the single-pass kernels blend through it
    int thr, gray_variant;
};
// *swapped = 1: the new model is in model_out (the caller exchanges the two buffers), 0: updated in place
int launch_asbl(const AsblLaunch &L, int nstreams, cudaStream_t stream, int *swapped);

// ---- MOG2 -------------------------------------------------------------------------------------
constexpr int MOG2_K = 5;             // nmixtures of the default-constructed cv::BackgroundSubtractorMOG2
constexpr int MOG2_PLANES = 5 * MOG2_K;   // per mode: weight, variance, mean B, G, R
constexpr int MOG2_TMAX = 32;         // frames per temporal batch launch
// Model state layout: tiles of 64 consecutive pixels; inside a tile the 25 planes are rows of 64 floats
// (plane q = mode*5 + {0 weight, 1 variance, 2 muB, 3 muG, 4 muR}).  A pixel's plane q sits q*64 floats
// after its plane 0 -- a compile-time offset -- and a warp that owns one tile reads / writes each plane as one
// contiguous 256-byte row.  Per pixel the footprint is the same 100 bytes as whole-frame planes.
constexpr int MOG2_TILE = 64;
constexpr int MOG2_TILE_FLOATS = MOG2_PLANES * MOG2_TILE;
__host__ __device__ inline size_t mog2_tile_off(size_t p) { return (p >> 6) * (size_t)MOG2_TILE_FLOATS + (p & 63); }

struct Mog2Launch {
    const uint8_t *frames;   // [S][T][npx*3]
    uint8_t *fg;             // [S][T][npx]
    uint8_t *bg;             // [S][T][npx*3] | [S][npx*3] | null
    float *state;            // [S][pstride/64 tiles][25][64]  (mog2_tile_off)
    uint8_t *nmodes;         // [S][pstride]
    size_t pstride;          // pixels per stream rounded up to whole tiles (64)
    // T == 1 production kernel only: the mask as bit-packed rows [S][h][wpr] (bit i of word k = pixel 32k+i), nullable.
    // The words must be zero on entry; the kernel sets the bits of the pixels whose mask byte is > bit_thr.  With `bits`
    // the byte mask `fg` may be null.
    unsigned *bits;
    size_t bits_stride;      // words per stream
    int w, wpr, bit_thr;
    int npx, T;
    int bg_last_only;
    int fresh;               // 1: state is uninitialised -> treat nmodes as 0 (first frame after create/reset)
    float one;               // 1.0f, opaque to the compiler: packed adds of products go through fma(p, one, b) because ptxas
                             // contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 whatever -fmad says (mog2_fastmath.cuh)
    int fast_ok;             // learning rates are inside the range the fast path's unguarded division is exact for
    int enable_thr, thr;
    int detect_shadows, shadow_value;
    float Tb, Tg, TB, varInit, varMin, varMax, tau;
    float alphaT[MOG2_TMAX];     // per-frame learning rate, 1-alphaT and prune = -lr*CT
    float alpha1[MOG2_TMAX];
    float prune[MOG2_TMAX];
};
int launch_mog2(const Mog2Launch &L, int nstreams, int variant, cudaStream_t stream);

}  // namespace bgsb
struct bgsb_ctx;
namespace bgsb {
// One frame per stream of the context's group, device buffers (what bgsb_process_dev does), for the pipeline: a MOG2
// context on its production kernel can emit the mask bit-packed into d_bits (zeroed by the caller; see Mog2Launch) and
// then needs no byte mask (d_fg may be null); every other context needs d_fg and leaves d_bits alone (*packed = 0).
int ctx_process_frame(bgsb_ctx *c, const uint8_t *d_frames, int w, int h, uint8_t *d_fg, uint8_t *d_bg, unsigned *d_bits,
                      int bit_thr, int *packed, int *fg_valid, int *bg_valid, cudaStream_t stream);
bool ctx_can_pack(const bgsb_ctx *c);
int ctx_nstreams(const bgsb_ctx *c);
int ctx_device(const bgsb_ctx *c);

// ---- DPZivkovicAGMMBGS (the reference's own adaptive GMM; state in the MOG2 tile layout, K <= 5) ----
struct DpzLaunch {
    const uint8_t *frame;    // [S] BGR frames, frame_stride bytes apart
    uint8_t *fg;             // [S] high-threshold masks, fg_stride bytes apart
    float *state;            // [S][pstride/64 tiles][25][64]
    uint8_t *nmodes;         // [S][pstride]
    size_t pstride, frame_stride, fg_stride;
    int npx, K;
    int fresh;               // InitModel: no modes yet
    float low_thr, alpha;    // params.LowThreshold() / Alpha() are floats (ZivkovicAGMM.h)
};
int launch_dpz(const DpzLaunch &L, int nstreams, cudaStream_t stream);

// ---- DPAdaptiveMedianBGS / DPMeanBGS / DPWrenGABGS (the DP package's simple per-pixel models, dp_simple.cu) ----
enum { DPS_MEDIAN = 0, DPS_MEAN = 1, DPS_WREN = 2 };
struct DpsLaunch {
    int kind;
    const uint8_t *frame;    // [S] BGR frames, frame_stride bytes apart
    uint8_t *fg;             // [S] high-threshold masks, fg_stride bytes apart
    float *state;            // Mean: [S][3][pstride] (mean B, G, R); WrenGA: [S][4][pstride] (mu B, G, R, var[0])
    uint8_t *median;         // AdaptiveMedian: [S][npx_frame * 3] 8-bit BGR model, median_stride bytes apart
    size_t pstride, frame_stride, fg_stride, median_stride;
    int npx;
    int fresh;               // InitModel: the model starts from this frame
    int update;              // AdaptiveMedian: this frame's Update() moves the model (frame_num % samplingRate == 1)
    unsigned high_u;         // AdaptiveMedian: (unsigned char)(2 * (unsigned char)threshold)
    float high_f;            // Mean: (float)(2u * threshold); WrenGA: 2 * (float)threshold
    float alpha, one_minus_alpha;
};
int launch_dp_simple(const DpsLaunch &L, int nstreams, cudaStream_t stream);

// ---- DPPratiMediodBGS (temporal medoid over a ring of sampled frames, dp_simple.cu) ----
// Per stream one block of `stream_bytes`: samples [H][3][plane1] u8 (planar B, G, R), medoid image [3][plane1] u8 (planar),
// distance sums [H][plane1] u16 stored per 4 pixels as (px0, px2 | px1, px3) (plane1 = padded pixels, plane3 = 3 * plane1:
// prati_layout); see dp_simple.cu.
struct PratiLaunch {
    const uint8_t *frame;    // [S] BGR frames, frame_stride bytes apart
    uint8_t *fg;             // [S] masks, fg_stride bytes apart
    uint8_t *state;          // [S] state blocks, stream_bytes apart
    size_t frame_stride, fg_stride, stream_bytes, plane3, plane1;
    int w, h, H;
    int n, pos;              // samples held so far / slot replaced once the ring is full (the same for every pixel)
    unsigned low, high;      // unsigned int members of PratiParams
};
inline void prati_layout(int npx, int H, size_t *plane3, size_t *plane1, size_t *stream_bytes)
{
    *plane1 = ((size_t)npx + 15) / 16 * 16;
    *plane3 = *plane1 * 3;
    *stream_bytes = (size_t)(H + 1) * *plane3 + (size_t)H * *plane1 * 2;
}
int launch_prati_subtract(const PratiLaunch &L, int nstreams, cudaStream_t stream);
int launch_prati_update(const PratiLaunch &L, int nstreams, cudaStream_t stream);

// ---- SigmaDeltaBGS (Lacassagne / Manzanera, the reference's sdLaMa091.cpp; dp_simple.cu) ----
struct SdLaunch {
    const uint8_t *frame;    // [S] BGR frames, frame_stride bytes apart
    uint8_t *fg;             // [S] masks, fg_stride bytes apart
    uint8_t *Mt, *Vt;        // [S] running median / variance images (interleaved like the frame), model_stride bytes apart
    size_t frame_stride, fg_stride, model_stride;
    int npx;                 // pixels of this launch
    int w;                   // frame width and ...
    long long p0;            // ... first pixel of this launch inside the frame (the initialiser's row rule needs positions)
    int first;               // no model yet: initialise from this frame, no mask
    unsigned N, vmin8, vmax8;    // amplification factor; minimal / maximal variance as the uint8_t helpers see them
};
int launch_sigma_delta(const SdLaunch &L, int nstreams, cudaStream_t stream);

// ---- morphology -------------------------------------------------------------------------------
int launch_morph_chain(const uint8_t *d_in, uint8_t *d_out, int w, int h, int nimages, const int *ops, int nops,
                       cudaStream_t stream);
// Any mix of byte and bit-packed masks ([nimages][h][(w+31)/32] words, bit i of word k = pixel 32k+i).
struct MorphIO {
    const uint8_t *in_bytes;     // exactly one of in_bytes / in_bits
    const unsigned *in_bits;
    uint8_t *out_bytes;          // either or both outputs
    unsigned *out_bits;
    int *parent;                 // with out_bits: the labeller's forest [nimages][w*h]; the output runs become its nodes
    int zero_border;             // ... after clearing the 1-px frame (nodes only; the stored words keep it)
    int max_ctas;                // > 0: cap on the grid (CTAs loop over the tiles); 0: one CTA per tile
};
int launch_morph_chain_io(const MorphIO &io, int w, int h, int nimages, const int *ops, int nops, cudaStream_t stream);

// ---- ingest: YUV 4:2:0 to dense BGR, as cv::cvtColor(COLOR_YUV2BGR_NV12 / _I420) (ingest/yuv420.cu) ----
struct Yuv420Launch {
    const uint8_t *y;        // first Y row of frame 0
    const uint8_t *u;        // first chroma row of frame 0: NV12 interleaved U,V; I420 the U plane
    const uint8_t *v;        // I420: first V row of frame 0 (unused for NV12)
    size_t y_pitch, c_pitch; // bytes between Y rows / chroma rows
    size_t src_frame_stride; // bytes between frames (the same for y, u and v)
    uint8_t *bgr;            // [nframes][rows][w][3], frames dst_frame_stride bytes apart
    size_t dst_frame_stride;
    int w, rows, nframes;    // w and rows even: rows / 2 chroma rows per frame
    int planar;              // 0 NV12, 1 I420
};
int launch_yuv420_to_bgr(const Yuv420Launch &L, cudaStream_t stream);

// ---- synthetic video ----------------------------------------------------------------------------
int launch_synth(uint8_t *d_frames, int nstreams, int T, int w, int h, int t0, uint32_t seed0,
                 cudaStream_t stream);
int launch_synth_churn(uint8_t *d_frames, int nstreams, int T, int w, int h, int t0, uint32_t seed0, cudaStream_t stream);

}  // namespace bgsb
