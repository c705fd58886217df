// Internal interface of the labeller (ccl.cu) for the other translation units of the library (pipeline.cu).
#pragma once
#include "common.cuh"

namespace bgsb {
struct CompRaw { int label, first_index, xmin, ymin, xmax, ymax, area, external; };
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
    // host round trips of the per-frame path: pinned staging (count + the first PIN_COMPS table rows, or moments) and
    // device buffers for the rectangle queries that live as long as the context (no allocator calls per frame)
    static constexpr int PIN_COMPS = 2048;
    uint8_t *h_pin = nullptr;               // 64 + PIN_COMPS * sizeof(CompRaw) bytes
    int *d_rects = nullptr;
    unsigned long long *d_mom = nullptr;
    int rect_cap = 0;
};

namespace bgsb {

// Label `nimages` bit-packed masks ([nimages][h][wpr] words, bit i of word k = pixel 32k+i of the row; bits beyond the
// row end must be zero).  zero_border: the 1-px frame counts as background (applied on the fly, the words are not
// modified).  The producer of the words must already have made every run start its own union-find root
// (ccl_init_word: the pack kernel and the morphology kernel do).
int ccl_label_bits(bgsb_ccl *c, const unsigned *d_bits, int w, int h, int nimages, int zero_border,
                   int32_t *d_labels, cudaStream_t stream);

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
