// Internal interface of the labeller (ccl.cu) for the other translation units of the library (pipeline.cu).
#pragma once
#include <vector>

#include "common.cuh"

namespace bgsb {
struct CompRaw { int label, first_index, xmin, ymin, xmax, ymax, area, external; };

// One rectangle of a batched cvMoments query: the image it lies in and its x, y, w, h (may cross the image edge), plus
// the tiling moment_tiles() fills in.
struct MomRec { int image, x, y, w, h, rows_per_tile, first_tile, pad; };

// Split the records' clipped rows into tiles of about equal work (one CTA each); -> the number of tiles.
int moment_tiles(MomRec *recs, int n, int w, int h);

// Host and device staging of a batched moments query, grown on demand (no allocator calls once large enough).
struct MomentBatch {
    MomRec *h_rec = nullptr, *d_rec = nullptr;          // pinned / device records
    unsigned long long *h_mom = nullptr, *d_mom = nullptr;   // pinned / device sums, 6 per record
    int cap = 0;
    int reserve(int n);
    void release();
    // h_rec[0, n) up, one moments launch over images of w x h -- byte masks [images][h][w] when mask != NULL, else
    // bit-packed {0,255} masks [images][h][wpr] -- and h_mom[0, 6n) down: m00 m10 m01 m20 m02 m11 per record
    // (ROI-relative, exact).  Asynchronous on `stream`.
    int enqueue(const uint8_t *mask, const unsigned *bits, int w, int h, int n, cudaStream_t stream);
};

// CvBlobDetectorCC::DetectNewBlob (blobdetect.cu) in two halves around the moments of step 4:
//   detect_rects : component table (raster order, every component) -> the rectangles step 4 weighs (external ones in
//                  reverse raster order, clustered and united), appended to `rects` as x, y, w, h
//   detect_finish: those rectangles with their moments (6 per rectangle) and the tracked blobs -> blob list, filters,
//                  top-10, track update and result; advances the detector
void detect_rects(const bgsb_blobdetector *bd, const bgsb_component *comps, int ncomp, int w, int h,
                  std::vector<int32_t> &rects);
void detect_finish(bgsb_blobdetector *bd, const int32_t *rects, int nrects, const uint64_t *mom, int w, int h,
                   const bgsb_blob *old_blobs, int n_old, bgsb_blob *new_blobs, int new_cap, int *n_new, int *result,
                   bgsb_blob *frame_blobs, int frame_cap, int *n_frame);
// The arguments of the batched entry points: S distinct non-NULL detectors whose "zeroBorder" equals the one the masks
// were labelled with, and per-stream old blob lists (old_blobs may be NULL: no tracked blobs).
int detect_check(bgsb_blobdetector *const *bds, int S, const bgsb_blob *const *old_blobs, const int *n_old,
                 int zero_border);
}

struct bgsb_ccl {
    int device = 0, max_w = 0, max_h = 0, max_images = 1;
    int w = 0, h = 0, nimages = 0;
    size_t img_px = 0, img_words = 0;      // per-image strides the work buffers were sized for
    int max_chunks = 0;                    // 256-word chunks per image at the largest geometry
    unsigned *d_bits = nullptr;            // bit-packed masks of the byte entry points (border already cleared)
    int *d_parent = nullptr;               // union-find forest, one slot per pixel, only run starts are used
    int *d_chunkcount = nullptr, *d_chunkprefix = nullptr;   // per image and 256-word chunk: roots, exclusive prefix
    int *d_done = nullptr;                 // [2][max_images] arrival counters of the roots / label kernels (zero between calls)
    int *d_ncomp = nullptr, *d_need_bg = nullptr;
    int table_images = 0;                  // images whose table rows the previous call may have filled
    int force_bg = 0;                      // 1: always run the background pass (A/B and tests)
    uint8_t *d_outer = nullptr, *d_mask_own = nullptr;
    int32_t *d_labels_own = nullptr;
    bgsb::CompRaw *d_comp = nullptr;
    int cap = 0;
    int coop_ctas = 0;                     // co-resident CTAs of the cooperative background kernel on this device
    int max_ctas = 0;                      // > 0: the labeller runs BESIDE another kernel (pipeline): background pass as plain
                                           // launches of at most this many CTAs instead of one cooperative launch
    bool dirty = false;                    // a call failed half-way: the arrival counters are cleared before the next one
    // what the moments are taken from: the byte masks of the last call, or its bit-packed masks (pipeline)
    const uint8_t *last_mask = nullptr;
    const unsigned *last_bits = nullptr;
    cudaStream_t last_stream = nullptr;
    cudaStream_t own_stream = nullptr;
    bool labelled = false;
    // host round trips of the per-frame path: pinned staging (count + the first PIN_COMPS table rows) and the
    // rectangle queries' buffers, which live as long as the context (no allocator calls per frame)
    static constexpr int PIN_COMPS = 2048;
    uint8_t *h_pin = nullptr;               // 64 + PIN_COMPS * sizeof(CompRaw) bytes
    bgsb::MomentBatch moments;
};

namespace bgsb {

// Label `nimages` bit-packed masks ([nimages][h][wpr] words, bit i of word k = pixel 32k+i of the row; bits beyond the
// row end must be zero).  zero_border: the 1-px frame counts as background (applied on the fly, the words are not
// modified).  The producer of the words must already have made every run start its own union-find root
// (ccl_init_word: the pack kernel and the morphology kernel do).
int ccl_label_bits(bgsb_ccl *c, const unsigned *d_bits, int w, int h, int nimages, int zero_border,
                   int32_t *d_labels, cudaStream_t stream);

// Pack [nimages][h][w] byte masks into [nimages][h][wpr] words with DetectNewBlob's threshold (a bit per byte > 128),
// frame kept, so that the words can go through the morphology kernel before labelling.
int ccl_pack_bytes(bgsb_ccl *c, const uint8_t *d_masks, unsigned *d_bits, int w, int h, int nimages, cudaStream_t stream);

// [nimages][(rows + 1) * 8] ints: per image {count, 0 x 7} then `rows` decoded bgsb_component rows (the first `rows`
// components in raster order); asynchronous on `stream`, which must be the stream of the labelling call.
int ccl_gather_tables(bgsb_ccl *c, int32_t *d_out, int rows, cudaStream_t stream);

#ifdef __CUDACC__
// the word as the labeller sees it: the 1-px image frame cleared when zero_border is set (OpenCV <= 3.1 cvFindContours)
__device__ __forceinline__ unsigned ccl_border(unsigned v, int y, int k, int w, int h, int wpr, int zero_border)
{
    if (zero_border) {
        if (y == 0 || y == h - 1) v = 0;
        if (k == 0) v &= ~1u;
        if (k == wpr - 1) v &= ~(1u << ((w - 1) & 31));
    }
    return v;
}
// every run start inside the (border-cleared) word becomes its own root; parent = this image's forest
__device__ __forceinline__ void ccl_init_word(int *parent, unsigned v, int base)
{
    unsigned s = v & ~(v << 1);
    while (s) {
        const int b = __ffs(s) - 1; s &= s - 1;
        parent[base + b] = base + b;
    }
}
#endif

}  // namespace bgsb
